"""world_size-2 gloo test of the sharded path's host logic (SURVEY.md 8e), on CPU.

The GPU engine shards contiguous row bands over ranks, every rank computes UN-normalised sums over
its own pixels with the global 1/N, and one all-reduce(sum) of [per-kernel statistics | loss
scalars | influence flags] makes every rank hold the 1-rank result.  Here the per-shard arithmetic is
done by the oracle (there is no GPU in this container); what is tested is the decomposition: band
bounds, the global normalisation, the packed exchange buffer, the OR of the influence flags."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import GOLDEN, ROOT


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import init_ref
    from oracle.graph import GraphCfg, PARAM_KEYS, graph_forward
    img = np.load(os.path.join(GOLDEN, "init_cases.npz"))["rgb_image"]          # 48 x 64 x 3
    H = img.shape[0]
    b0, b1 = H * rank // world, H * (rank + 1) // world                          # the engine's band rule
    mus, A = init_ref.kernel_grid([6, 8], 2, False)
    nu, ga = init_ref.experts(img, mus)
    K = mus.shape[0]
    p = {"pis": torch.tensor(init_ref.pis(K, True), dtype=torch.float64), "musX": torch.tensor(mus),
         "A_diagonal": torch.tensor(A), "A_corr": torch.zeros(K, 2, 2, dtype=torch.float64),
         "gamma_e": torch.tensor(ga), "nu_e": torch.tensor(nu, dtype=torch.float64)}
    jd = init_ref.gen_domain(img, 2)
    cfg = GraphCfg(dim_domain=2, num_channels=3, use_determinant=True, train_inverse_cov=False, use_yuv=False, start_pis=K)

    def grads(rows, scale):
        leaf = {k: v.clone().requires_grad_(True) for k, v in p.items()}
        d = torch.tensor(jd[rows].reshape(-1, 5).astype(np.float32).astype(np.float64))
        out = graph_forward(leaf, np.ones(K, bool), d[:, :2], d[:, 2:], cfg)
        # the graph's loss is a MEAN over the fed pixels; a shard contributes sum/N_total = mean * n_shard/N
        g = torch.autograd.grad(out["loss"] * scale, [leaf[k] for k in PARAM_KEYS], allow_unused=True)
        flat = torch.cat([(torch.zeros_like(leaf[k]) if gi is None else gi).reshape(-1) for k, gi in zip(PARAM_KEYS, g)])
        return flat, float(out["loss"].detach()) * scale, out["kernel_list_batch"].to(torch.float64)

    n_band = b1 - b0
    flat, loss_part, infl = grads(slice(b0, b1), n_band / H)
    xbuf = torch.cat([flat, torch.tensor([loss_part], dtype=torch.float64), infl])   # one packed buffer
    dist.all_reduce(xbuf)
    if rank == 0:
        ref_flat, ref_loss, ref_infl = grads(slice(0, H), 1.0)
        np.save(os.path.join(out_dir, "sharded.npy"), xbuf.numpy())
        np.save(os.path.join(out_dir, "single.npy"), torch.cat([ref_flat, torch.tensor([ref_loss], dtype=torch.float64), ref_infl]).numpy())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_row_band_sharding_equals_single_rank(tmp_path, world):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    a = np.load(str(tmp_path / "sharded.npy"))
    b = np.load(str(tmp_path / "single.npy"))
    K = 48
    ng = a.size - 1 - K
    np.testing.assert_allclose(a[:ng], b[:ng], rtol=1e-9, atol=1e-16)
    assert abs(a[ng] - b[ng]) < 1e-12
    np.testing.assert_array_equal(a[ng + 1:] > 0, b[ng + 1:] > 0)          # influence flags: OR over ranks


def test_band_bounds_cover_every_row_once():
    for H in (135, 1080, 720, 7):
        for world in (1, 2, 3, 4, 8):
            bands = [(H * r // world, H * (r + 1) // world) for r in range(world)]
            assert bands[0][0] == 0 and bands[-1][1] == H
            assert all(bands[i][1] == bands[i + 1][0] for i in range(world - 1))


def _ssim_map(a, b, nd):
    """Per-position SSIM map (VALID) of two already padded arrays, float64 (oracle/ssim.py pieces)."""
    from oracle import ssim as ossim
    win = ossim.gauss_window(nd, dtype=np.float64)
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    m0, m1 = ossim._reduce_valid(a, win), ossim._reduce_valid(b, win)
    num0, den0 = 2 * m0 * m1, m0 * m0 + m1 * m1
    lum = (num0 + c1) / (den0 + c1)
    cs = (2 * ossim._reduce_valid(a * b, win) - num0 + c2) / (ossim._reduce_valid(a * a + b * b, win) - den0 + c2)
    return lum * cs


def _ssim_shard_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    rs = np.random.RandomState(3)
    H, W, C = 46, 52, 3
    res = rs.uniform(0, 1, (H, W, C))
    tgt = np.clip(res + 0.1 * rs.standard_normal((H, W, C)), 0, 1)
    # the product's scheme (Smoe._init_halo / smoe_ssim_loss with a region): the rank's buffer is its block plus a ring
    # of 10 pixels clipped to the image; SYMMETRIC padding at the buffer's borders; only the block's positions count
    lo, hi = H * rank // world, H * (rank + 1) // world
    blo, bhi = max(lo - 10, 0), min(hi + 10, H)
    pad = ((5, 5), (5, 5), (0, 0))
    m = _ssim_map(np.pad(res[blo:bhi], pad, mode="symmetric"), np.pad(tgt[blo:bhi], pad, mode="symmetric"), 2)
    part = torch.tensor(m[lo - blo:hi - blo].sum(axis=(0, 1)))
    dist.all_reduce(part)
    full = _ssim_map(np.pad(res, pad, mode="symmetric"), np.pad(tgt, pad, mode="symmetric"), 2).sum(axis=(0, 1))
    if rank == 0:
        np.save(os.path.join(out_dir, "ssim.npy"), np.stack([part.numpy(), full]))
    dist.destroy_process_group()


def test_sharded_ssim_region_scheme_equals_full_image(tmp_path):
    """Sum over ranks of (SSIM values of the rank's own positions, computed on block + 10-pixel ring with symmetric
    padding at the ring's borders) == SSIM sum of the whole image: a window centred within the block reaches at most 5
    pixels out, and the padding is only ever consulted at true image borders."""
    import torch.multiprocessing as mp
    mp.spawn(_ssim_shard_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    part, full = np.load(os.path.join(str(tmp_path), "ssim.npy"))
    np.testing.assert_allclose(part, full, rtol=1e-12)


@pytest.mark.parametrize("shape,k,world", [((1080, 1920, 3), [128, 256], 8), ((1080, 1920, 3), [128, 256], 4),
                                           ((720, 1280, 32, 3), [32, 64, 32], 8), ((135, 96, 3), [12, 10], 2),
                                           ((40, 48, 12, 3), [4, 4, 3], 3), ((33, 47, 1), [4, 4], 5)])
def test_block_decomposition_covers_every_pixel_once(shape, k, world):
    """Host logic of the pixel sharding (Smoe._choose_blocks): one rectangle per rank, disjoint, covering the image,
    cuts on the tile grid when the image is large enough; 2x4 blocks (not 8 bands) for config 3 on 8 ranks."""
    sys.path.insert(0, ROOT)
    from smoe_b200 import Smoe
    s = object.__new__(Smoe)
    s.image = np.zeros(shape, np.float32)
    s.dim_domain = len(shape) - 1
    s.train_inverse_cov = False
    s.generate_kernel_grid(k)
    blocks = s._choose_blocks(world)
    assert len(blocks) == world and int(np.prod(s._block_grid)) == world
    cover = np.zeros(shape[:-1], np.int32)
    for blk in blocks:
        assert all(hi > lo for lo, hi in blk)
        cover[tuple(slice(lo, hi) for lo, hi in blk)] += 1
    assert (cover == 1).all()
    if shape[:2] == (1080, 1920) and world == 8:
        assert tuple(s._block_grid) == (2, 4)
        assert all((lo % 16 == 0) for blk in blocks for lo, _ in blk[:1]) and all((blk[1][0] % 32 == 0) for blk in blocks)
