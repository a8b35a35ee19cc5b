"""The tile runner without a GPU: pipeline2d.run_tiles (the batch loop of every predictor) and pipeline2d.predict_tiles
(the plain or test-time-augmented step) driven by a fake engine that records every forward."""
import pytest
import torch

from bio_image_unet_b200 import pipeline2d as P


class FakeEngine:
    """Engine.forward's contract on the CPU: exactly `batch` (+ n_per with the shared Siam encoder) input tiles. The
    outputs identify their inputs: u8 is the current tile, val = current + 1000 * previous tile (previous: the second
    input, or tile j of the shared window for pair j)."""

    def __init__(self, batch, n_per=0):
        self.batch, self.n_per = batch, n_per
        self.calls, self.outs = [], []

    def forward(self, tiles, tiles_prev=None, want_val=False, want_u8=True):
        assert tiles.is_contiguous() and tiles.shape[0] == self.batch + self.n_per
        assert tiles_prev is None or (tiles_prev.is_contiguous() and tiles_prev.shape[0] == self.batch)
        self.calls.append(dict(tiles=tiles.clone(), prev=None if tiles_prev is None else tiles_prev.clone(),
                               want_val=want_val, want_u8=want_u8))
        cur = tiles[self.n_per:]
        prev = tiles_prev if tiles_prev is not None else (tiles[:self.batch] if self.n_per else None)
        val = cur.float() + (0 if prev is None else 1000 * prev.float())
        out = (val if want_val else None, cur.clone() if want_u8 else None)
        self.outs.append(out)
        return out


def tiles_of(n, offset=1):
    """n uint8 tiles (n, 1, 2, 3), tile i filled with i + offset (never 0, so zero padding is visible)."""
    return (torch.arange(n, dtype=torch.uint8) + offset).view(n, 1, 1, 1).expand(n, 1, 2, 3).contiguous()


def check_batches(eng, src, tile_batch, n_per=0, prev=None):
    """Every forward got the window of its batch, zero-padded to tile_batch (+ n_per) tiles."""
    n = src.shape[0] - n_per
    starts = list(range(0, n, tile_batch))
    assert len(eng.calls) == len(starts)
    for call, s in zip(eng.calls, starts):
        cnt = min(tile_batch, n - s)
        t = call['tiles']
        assert t.shape[0] == tile_batch + n_per
        assert torch.equal(t[:cnt + n_per], src[s:s + cnt + n_per])
        assert not t[cnt + n_per:].any()
        if prev is not None:
            assert torch.equal(call['prev'][:cnt], prev[s:s + cnt]) and not call['prev'][cnt:].any()


@pytest.mark.parametrize('n,tile_batch', [(7, 3), (6, 3), (4, 4), (3, 8), (1, 1)])
def test_plain_batches(n, tile_batch):
    tiles = tiles_of(n)
    eng = FakeEngine(tile_batch)
    u8, val = P.run_tiles(eng, tiles, tile_batch)
    check_batches(eng, tiles, tile_batch)
    assert val is None and torch.equal(u8, tiles)
    assert all(c['want_u8'] and not c['want_val'] for c in eng.calls)


@pytest.mark.parametrize('want_u8', [True, False])
def test_float_output(want_u8):
    tiles = tiles_of(10)
    eng = FakeEngine(4)
    u8, val = P.run_tiles(eng, tiles, 4, want_val=True, want_u8=want_u8)
    check_batches(eng, tiles, 4)
    assert torch.equal(val, tiles.float())
    assert torch.equal(u8, tiles) if want_u8 else u8 is None
    assert all(c['want_val'] and c['want_u8'] == want_u8 for c in eng.calls)


def test_single_batch_is_not_copied():
    tiles = tiles_of(5)
    eng = FakeEngine(5)
    u8, val = P.run_tiles(eng, tiles, 5, want_val=True)
    assert u8.data_ptr() == eng.outs[0][1].data_ptr() and val.data_ptr() == eng.outs[0][0].data_ptr()


@pytest.mark.parametrize('n,tile_batch', [(7, 3), (6, 6), (2, 5)])
def test_two_input_siam(n, tile_batch):
    cur, prev = tiles_of(n), tiles_of(n, offset=100)
    eng = FakeEngine(tile_batch)
    u8, val = P.run_tiles(eng, cur, tile_batch, prev_tiles=prev, want_val=True)
    check_batches(eng, cur, tile_batch, prev=prev)
    assert torch.equal(u8, cur) and torch.equal(val, cur.float() + 1000 * prev.float())


@pytest.mark.parametrize('n_pairs,n_per,tile_batch', [(8, 2, 3), (6, 3, 6), (4, 1, 4), (2, 4, 5)])
def test_shared_encoder_windows(n_pairs, n_per, tile_batch):
    """Pair j = (tile j, tile j + n_per): the batch at pair s takes tiles[s : s + cnt + n_per], so windows of
    consecutive batches overlap by n_per tiles."""
    tiles_u = tiles_of(n_pairs + n_per)
    eng = FakeEngine(tile_batch, n_per)
    u8, val = P.run_tiles(eng, tiles_u, tile_batch, n_per=n_per, want_val=True)
    check_batches(eng, tiles_u, tile_batch, n_per=n_per)
    assert u8.shape[0] == n_pairs
    assert torch.equal(u8, tiles_u[n_per:])
    assert torch.equal(val, tiles_u[n_per:].float() + 1000 * tiles_u[:n_pairs].float())


@pytest.mark.parametrize('n_per', [0, 2])
def test_on_val_streaming(n_per):
    tiles = tiles_of(11 + n_per)
    eng = FakeEngine(4, n_per)
    got = []
    assert P.run_tiles(eng, tiles, 4, n_per=n_per, on_val=lambda s, v: got.append((s, v))) == (None, None)
    check_batches(eng, tiles, 4, n_per=n_per)
    assert [(s, v.shape[0]) for s, v in got] == [(0, 4), (4, 4), (8, 3)]
    want = tiles[n_per:].float() + (1000 * tiles[:11].float() if n_per else 0)
    assert torch.equal(torch.cat([v for _, v in got]), want)
    assert all(c['want_val'] and not c['want_u8'] for c in eng.calls)


def test_progress_wraps_batch_starts():
    seen = []

    def progress(it):
        seen.append(list(it))
        return it
    P.run_tiles(FakeEngine(3), tiles_of(8), 3, progress=progress)
    assert seen == [[0, 3, 6]]


def _no_merge(*a, **k):
    raise AssertionError('the plain path must not reach the test-time augmentation merge')


@pytest.mark.parametrize('out_dtype', [torch.uint8, torch.float32])
def test_plain_step_comes_straight_from_the_net(monkeypatch, out_dtype):
    monkeypatch.setattr(P.E, 'tta_accumulate', _no_merge)
    tiles = tiles_of(7)
    eng = FakeEngine(3)
    asked = []

    def gather(t):
        asked.append(t)
        return tiles
    want_u8 = out_dtype == torch.uint8
    res, plain = P.predict_tiles(gather, lambda tl, on_val: P.run_tiles(eng, tl, 3, want_val=not want_u8,
                                                                        want_u8=want_u8, on_val=on_val),
                                 7, None, 2, out_dtype=out_dtype)
    assert asked == [0] and plain is tiles
    assert torch.equal(res, tiles if want_u8 else tiles.float())
    assert all(c['want_u8'] == want_u8 and c['want_val'] != want_u8 for c in eng.calls)


@pytest.mark.parametrize('codes', [[0, 1, 2, 3], [0]])
@pytest.mark.parametrize('out_dtype', [torch.uint8, torch.float32])
def test_augmented_step(monkeypatch, codes, out_dtype):
    """Every pass gathers its transform in order and streams every batch into the merge at its start; the last pass
    writes the chunk's result buffer; the plain tiles returned are gather(0)."""
    merges = []

    def merge(val, acc, dims, t, p, passes, out_u8=None, out_f32=None):
        out = out_u8 if out_dtype == torch.uint8 else out_f32
        assert (out_f32 if out_dtype == torch.uint8 else out_u8) is None
        assert acc is None if passes == 1 else acc.shape == val.shape
        assert out.shape == val.shape
        merges.append((t, p, passes, dims, val.shape[0]))
        if p == passes - 1:
            out.copy_(val)
    monkeypatch.setattr(P.E, 'tta_accumulate', merge)
    n, tb = 10, 4
    eng = FakeEngine(tb)
    gathered = {}

    def gather(t):
        gathered[t] = tiles_of(n, offset=1 + 20 * t)
        return gathered[t]
    res, plain = P.predict_tiles(gather, lambda tl, on_val: P.run_tiles(eng, tl, tb, on_val=on_val), n, codes, 2,
                                 out_dtype=out_dtype)
    assert list(gathered) == codes and plain is gathered[0]
    k = len(codes)
    assert merges == [(t, p, k, 2, cnt) for p, t in enumerate(codes) for cnt in (4, 4, 2)]
    assert res.dtype == out_dtype and torch.equal(res.float(), gathered[codes[-1]].float())
