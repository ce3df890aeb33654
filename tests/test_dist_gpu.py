"""2-rank NCCL test of the PRODUCT path (needs >= 2 GPUs; skipped on a 1-GPU box): two ranks each run the fused step
of avatarclip_b200.trainer on the view avatarclip_b200.dist.view_index assigns them (tcgen05 engine), all-reduce the
flat gradient over NCCL and apply the fused Adam with grad_scale 1/2; the result must equal ONE rank accumulating the
two views' gradients and applying the same Adam (SURVEY.md 8e: N ranks x 1 view == 1 rank x N views)."""
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu


def _world(device, pg=None):
    from avatarclip_b200 import workload as WL
    from avatarclip_b200.clip_vit import ClipImageTower
    from avatarclip_b200.trainer import AppearanceTrainer
    sp, cp = WL.synth_states(WL.S_SDF_KW, WL.S_COL_KW, seed=0)
    _, _, _, ren = WL.build_networks(WL.S_SDF_KW, WL.S_COL_KW, WL.S_REN_KW, sp, cp, 0.3, device, engine=1)
    tower = ClipImageTower(WL.random_vit_state(seed=0), device=device)
    text = torch.randn(2, 512, generator=torch.Generator().manual_seed(5))
    return AppearanceTrainer(ren, tower, text, lr=5e-4, process_group=pg, device=device)


def _view(i):
    from avatarclip_b200.workload import make_view
    return make_view(i, n_rays=160, H=96, W=96, seed=0, bg_choice=3)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    from avatarclip_b200 import dist as ad
    from avatarclip_b200.trainer import DeviceView
    pg = ad.init_from_env("nccl", dev)
    tr = _world(dev, pg)
    g1 = None
    for step in range(2):
        tr.step(DeviceView(_view(ad.view_index(step, rank, world)), dev))
        if step == 0:
            g1 = tr.grad.clone()          # after the all-reduce: the sum over both ranks' views
    torch.cuda.synchronize()
    if rank == 0:
        torch.save({"flat": tr.fp.flat.cpu(), "grad1": g1.cpu()}, out)
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_product_step_equals_two_view_accumulation(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "r0.pt")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    # ---- one rank, two views accumulated per optimiser step, same fused Adam with grad_scale 1/2
    import ctypes as C
    from avatarclip_b200 import _lib, dist as ad
    from avatarclip_b200.trainer import DeviceView
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    tr = _world(dev)
    acc1 = None
    for step in range(2):
        acc = torch.zeros_like(tr.grad)
        for r in range(2):
            acc += tr.forward_backward(DeviceView(_view(ad.view_index(step, r, 2)), dev))
        if step == 0:
            acc1 = acc.clone()
        tr.iter_step += 1
        _lib.check(_lib.lib().avc_adam_step(_lib.ptr(tr.fp.flat), _lib.ptr(acc), _lib.ptr(tr.exp_avg),
                                            _lib.ptr(tr.exp_avg_sq), tr.fp.n, tr.lr, 0.9, 0.999, tr.eps, tr.iter_step,
                                            0.5, _lib.stream_ptr()), "avc_adam_step")
    torch.cuda.synchronize()
    want = tr.fp.flat.cpu()
    # run-to-run noise of ONE rank on identical inputs (fp32 atomics in the split-K CLIP GEMMs and the weight-gradient
    # tiles land in a different order every run; the CLIP tower rounds to fp16 after them): the yardstick for g_err
    tr2 = _world(dev)
    rep = torch.zeros_like(tr2.grad)
    for r in range(2):
        rep += tr2.forward_backward(DeviceView(_view(ad.view_index(0, r, 2)), dev))
    torch.cuda.synchronize()
    noise = (rep.cpu() - acc1.cpu()).norm().item() / acc1.cpu().norm().item()
    g_err = (got["grad1"] - acc1.cpu()).norm().item() / acc1.cpu().norm().item()
    p_err = (got["flat"] - want).abs().max().item()
    print(f"2-rank NCCL vs 2-view accumulation: first-step summed-gradient rel-L2 {g_err:.3e} (single-rank repeat noise "
          f"{noise:.3e}), max parameter diff after 2 steps {p_err:.3e}")
    import util_neus as U
    U.log_parity("nccl_2rank_product", {"grad_rel_l2": g_err, "repeat_noise_rel_l2": noise, "max_param_diff": p_err})
    # same weights, same views: what differs is the order of fp32 atomics (measured 1.6e-4, the level two runs of one rank
    # differ by); the bar is the gradient-parity bar of the NeuS tests
    assert g_err < 1e-3
    # two Adam steps of lr 5e-4 (measured 7.3e-4): Adam's sign-like first updates turn last-bit gradient differences of
    # near-zero coordinates into differences of the order of lr; bounded by the 2 x lr the two steps can move a coordinate
    assert p_err < 1.1e-3
