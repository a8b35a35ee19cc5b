"""torchrun worker: unet.Predict, siam_unet.Predict and unet3d.Predict with blend='gaussian' and distributed=True must
reproduce the single-process result exactly.

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29537 tests/run_dist_blend.py OUTDIR
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bio_image_unet_b200 import tiff  # noqa: E402


def main(out_dir):
    rank, local = int(os.environ['RANK']), int(os.environ['LOCAL_RANK'])
    world = int(os.environ['WORLD_SIZE'])
    if torch.cuda.device_count() >= world:
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    else:       # 1-GPU box: both ranks share cuda:0, collectives go through gloo
        local = local % torch.cuda.device_count()
        torch.cuda.set_device(local)
        dist.init_process_group('gloo')
    from bio_image_unet_b200.siam_unet import Predict as PredictSiam
    from bio_image_unet_b200.siam_unet.siam_unet import Siam_UNet
    from bio_image_unet_b200.unet import Predict as PredictUnet
    from bio_image_unet_b200.unet import Unet
    from bio_image_unet_b200.unet3d import Predict as Predict3D
    from bio_image_unet_b200.unet3d import UNet3D
    ok = True

    def compare(name, make, kw):
        nonlocal ok
        res_d = os.path.join(out_dir, f'{name}_dist.tif')
        make(res_d, dict(kw, distributed=True))
        dist.barrier()
        if rank == 0:
            res_s = os.path.join(out_dir, f'{name}_single.tif')
            make(res_s, dict(kw, device=f'cuda:{local}'))
            same = np.array_equal(tiff.imread(res_d), tiff.imread(res_s))
            print(f'[dist] {name} blend=gaussian: distributed == single: {same}')
            ok &= bool(same)

    torch.manual_seed(3)
    ckpt = os.path.join(out_dir, f'unet_{rank}.pt')
    torch.save({'state_dict': Unet(n_filter=8).state_dict(), 'n_filter': 8, 'in_channels': 1, 'out_channels': 1}, ckpt)
    imgs = np.random.default_rng(7).integers(0, 3000, (7, 90, 70)).astype('uint16')
    for mode in ('single', 'all'):
        compare(f'unet_{mode}', lambda res, kw: PredictUnet(imgs.copy(), res, ckpt, **kw),
                dict(resize_dim=(64, 64), add_tile=1, normalization_mode=mode, show_progress=False, precision='bf16',
                     blend='gaussian'))
    torch.manual_seed(2)
    ckpt = os.path.join(out_dir, f'siam_{rank}.pt')
    torch.save({'state_dict': Siam_UNet(n_filter=8, mode='concat').state_dict(), 'n_filter': 8, 'mode': 'concat'}, ckpt)
    movie = np.random.default_rng(4).integers(0, 2000, (7, 40, 52)).astype('uint16')
    compare('siam', lambda res, kw: PredictSiam(movie, res, ckpt, **kw),
            dict(resize_dim=(32, 32), add_tile=1, show_progress=False, precision='bf16', blend='gaussian'))
    torch.manual_seed(5)
    ckpt = os.path.join(out_dir, f'u3d_{rank}.pt')
    torch.save({'state_dict': UNet3D(n_filter=4).state_dict(), 'n_filter': 4, 'in_channels': 1, 'out_channels': 1}, ckpt)
    vol = np.random.default_rng(11).integers(0, 3000, (44, 40, 48)).astype('uint16')
    for add_patch in (1, 0):
        compare(f'u3d{add_patch}', lambda res, kw: Predict3D(vol.copy(), res, ckpt, **kw),
                dict(resize_dim=(8, 16, 16), add_patch=add_patch, progress_bar=False, precision='bf16',
                     blend='gaussian'))
    flag = torch.tensor([1 if ok else 0], device='cuda' if dist.get_backend() == 'nccl' else 'cpu')
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    if rank == 0:
        open(os.path.join(out_dir, 'DIST_OK' if ok else 'DIST_FAIL'), 'w').write('done')
    sys.exit(0 if flag.item() == 1 else 1)


if __name__ == '__main__':
    main(sys.argv[1])
