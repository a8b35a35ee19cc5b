"""Every op of the Siam_UNet, Unet_v0, MultiOutputUnet and U-Net++ layer programs against the exact single-op reference.

The machinery (program mirror, references, stop-point reruns) is that of tests/test_gpu_layer_exact.py; this module
adds the cases of the families whose ops and buffer layouts the Unet / AttentionUnet / 3D cases do not reach:

- Siam_UNet's twin-encoder buffers: [current | previous], or with the shared encoder the unique tiles, previous
  stream = images [0, B), current stream = images [N, N + B); the concat join's two pools into 'joincat'; the max join
  (bit-exact) and the depth-wise cross-correlation (its own interval, sequential fp32 sums of up to h * w taps);
- Unet_v0's ReLU blocks, its skip taken after the first conv, decode9 and the 1 -> 1 head;
- MultiOutputUnet's float32 input, which always takes the CUDA-core first conv;
- U-Net++'s shared per-level buffers: multi-segment concat prefixes at channel offsets upw[l] + k pc[l], bilinear
  x2 up-sampling (align_corners=True) into one slot that every node of a level reuses, and a first conv of every node
  that writes the same v{l}. Only the last node of each level survives the forward; the others are checked after a
  forward that stops after them.
"""
import pytest

from tests.test_gpu_layer_exact import KNOBS, PRECISIONS, _record, kernel_knob, run_case  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu

HEADS_MO = (('a', 1, 'sigmoid'), ('b', 2, 'none'), ('c', 1, 'tanh'))

CASES = {
    # corr at level-4 extents 4 x 4 (even: the extra 'same' padding at the far end of both axes)
    'siam_corr_nf16_64x64': dict(kind='siam2d', siam_mode='corr', nf=16, tile=(64, 64), batch=2),
    # 5 x 3: odd and non-square
    'siam_corr_nf16_80x48': dict(kind='siam2d', siam_mode='corr', nf=16, tile=(80, 48), batch=2),
    # 32 x 32: 1024 taps per output, channel groups of G = 8 in shared memory
    'siam_corr_nf16_512x512': dict(kind='siam2d', siam_mode='corr', nf=16, tile=(512, 512), batch=1),
    # 64 x 64: 4096 taps, G = 2
    'siam_corr_nf16_1024x1024': dict(kind='siam2d', siam_mode='corr', nf=16, tile=(1024, 1024), batch=1),
    # element-wise maximum of the two embeddings, bit-exact
    'siam_max_nf16_128x128': dict(kind='siam2d', siam_mode='max', nf=16, tile=(128, 128), batch=2),
    # both streams pooled into joincat [current | previous], conv_concat reads the two halves
    'siam_concat_nf32_128x128': dict(kind='siam2d', siam_mode='concat', nf=32, tile=(128, 128), batch=2),
    # the previous frame is ignored: one stream, Unet's program
    'siam_control_nf16_128x128': dict(kind='siam2d', siam_mode='control', nf=16, tile=(128, 128), batch=2),
    # shared encoder, N = 2 tiles per frame against B = 3 pairs: current stream = images [2, 5), previous = [0, 3)
    'siam_corr_shared_nf16_64x128': dict(kind='siam2d', siam_mode='corr', nf=16, tile=(64, 128), batch=3,
                                         siam_shared=2),
    'siam_concat_shared_nf16_64x128': dict(kind='siam2d', siam_mode='concat', nf=16, tile=(64, 128), batch=3,
                                           siam_shared=2),
    # ReLU blocks, skip after the first conv, decode9 + the 1 -> 1 head; row-kernel widths
    'unet_v0_nf16_64x128': dict(kind='unet2d_v0', nf=16, tile=(64, 128), batch=2),
    'unet_v0_nf32_48x144': dict(kind='unet2d_v0', nf=32, tile=(48, 144), batch=1),
    # float32 tiles (CUDA-core first conv, no / 255), three heads with sigmoid / none / tanh
    'mo2d_nf16_64x128': dict(kind='mo2d', nf=16, tile=(64, 128), batch=2, heads=HEADS_MO, float_input=True),
    # U-Net++ 4 levels: ragged level extents (64 x 96 -> 4 x 6)
    'nested_nf16_64x96': dict(kind='nested2d', nf=16, tile=(64, 96), batch=2, heads=HEADS_MO),
    # deepest extent 1 (16 x 32 -> 1 x 2): bilinear from a single source row, CUDA-core fallback of the small planes
    'nested_nf16_16x32': dict(kind='nested2d', nf=16, tile=(16, 32), batch=2, heads=HEADS_MO),
    # the wide levels on the tensor-core kernels, bilinear from extent 64
    'nested_nf32_128x128': dict(kind='nested2d', nf=32, tile=(128, 128), batch=1, heads=HEADS_MO),
    # U-Net++ 3 levels, and its deepest extent 1 (8 x 16 -> 1 x 2)
    'nested3l_nf16_64x96': dict(kind='nested2d_3l', nf=16, tile=(64, 96), batch=2, heads=HEADS_MO),
    'nested3l_nf16_8x16': dict(kind='nested2d_3l', nf=16, tile=(8, 16), batch=2, heads=HEADS_MO),
}


@pytest.mark.parametrize('knob', KNOBS)
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case', list(CASES))
def test_family_layers_exact(case, precision, knob, kernel_knob):
    rows_on = kernel_knob(knob)
    _record(precision, run_case(precision=precision, rows_on=rows_on, **CASES[case]))


@pytest.mark.parametrize('case', list(CASES))
def test_family_layers_exact_fp32(case):
    """fp32 on the CUDA-core kernels (every conv, head and transposed conv reports the fallback bit)."""
    from tests.test_gpu_layer_exact import CONV, HEAD, UP, program
    res = run_case(precision='fp32', **CASES[case])
    spec = CASES[case]
    ops = program(spec['kind'], spec['nf'], False, spec.get('siam_mode', 'concat'))[1]
    assert all(k & 16 for k, o in zip(res['kinds'], ops) if o['kind'] in (CONV, HEAD, UP))
    _record('fp32', res)
