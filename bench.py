#!/usr/bin/env python
"""bench.py -- appearance-optimisation steps/s (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): one train_clip step = render 512 rays x (64+64) samples through the 8x256
SDF + 4x256 colour MLPs (placement + fine pass), shading/canvas/losses on a 224x224 canvas, CLIP ViT-B/32 on the
texture and the shading canvas, full backward (second-order SDF terms included) and Adam.  Synthetic data:
seeded geometric-init weights, seeded random CLIP weights (the real ViT-B-32.pt is not on disk), disc-shaped
silhouettes (avatarclip_b200/workload.py).

N > 1: one camera view per rank per step (weak scaling), one NCCL all-reduce of the flat fp32 gradient per step.

Native arm JSON keys follow the driver contract; see DESIGN.md "Measurement" for how each number is taken.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from avatarclip_b200 import workload as WL  # noqa: E402  (host-side numpy / CPU torch only)

METRIC = "appearance-optim steps/sec (512 rays x 128 samples, CLIP loss)"
# config.workload of BOTH arms (the native line and `--impl reference`): the same string, so the two lines name one workload
WORKLOAD = ("BASELINE configs[1]: 512 rays x (64+64) samples, 8x256 SDF + 4x256 colour, "
            "CLIP ViT-B/32 loss on 2 canvases 224x224, Adam; 1 view per GPU per step")
# dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu (profiles/r2_launches_tcgen05_engine.txt, final round-2
# build): mean over the 41 NT / 21 TN launches of one step (all in the fine pass; 11.1 GB of DRAM traffic per step in total)
TRAFFIC_PER_LAUNCH = {"avc::tc::gemm_tc_tn_kernel": 128.0e6, "avc::tc::gemm_tc_nt_kernel": 188.6e6}
N_RAYS, CANVAS = 512, 224
SDF_KW, COL_KW, REN_KW = WL.B2_SDF_KW, WL.B2_COL_KW, WL.B2_REN_KW
VARIANCE = 0.3
PARITY_JITTER_SEED = 1234
CLIP_WEIGHT_BYTES_PER_PASS = 87_849_216 * 2      # fp16 ViT-B/32 image tower, read once per pass (fwd, input-grad bwd)


def nt_designed_bytes_per_step():
    """HBM bytes the NT launches of one step move BY DESIGN (unfused layers: every linear reads its split operand and
    its stashed epilogue operands and writes its outputs once), B2 config, in units of one 256-wide fp32 row (1 KB):
    fine pass per point: value 8 layers (reads 7.16, writes sp' stash + split 16), features 2, gradient chain 7 x 3
    + 1.3, colour 4 x 2 + 1, colour dgrad 3 x 2.5 + 1 + 2, second-order sweep 8 x 5, value dgrad 8 x 4;
    placement passes per point: 8 layers, split in / split out (15.16)."""
    fine = 23.16 + 2 + 21 + 1.3 + 9 + 8.5 + 2 + 40 + 32
    place = 15.16
    p_fine = N_RAYS * (REN_KW["n_samples"] + REN_KW["n_importance"])
    p_place = N_RAYS * (REN_KW["n_samples"] + 3 * REN_KW["n_importance"] // 4)
    return 1024.0 * (fine * p_fine + place * p_place)


def algorithmic_flops_per_step():
    """SURVEY.md 8d: (6.875 F_sdf + 3 F_col) per fine sample point, F = 2*MAC; + CLIP fwd+dgrad for two images.
    Returns (all MLP FLOP, the part executed by the NT tiles, the part executed by the TN (weight-gradient) tiles,
    CLIP FLOP).  NT: value fwd 1 + gradient chain 1 + placement passes 0.875 + value dgrad 1 + second-order sweep 1
    = 4.875 F_sdf, colour fwd + dgrad = 2 F_col.  TN: 2 F_sdf + 1 F_col."""
    mac_sdf = 39 * 256 + 6 * 256 * 256 + 256 * 217 + 256 * 257        # 9 linears of the 8x256 net
    mac_col = 262 * 256 + 3 * 256 * 256 + 2 * 3 * 256                 # 4x256 + two 3-wide heads
    pts = N_RAYS * (REN_KW["n_samples"] + REN_KW["n_importance"])
    mlp = (6.875 * 2 * mac_sdf + 3 * 2 * mac_col) * pts
    nt = (4.875 * 2 * mac_sdf + 2 * 2 * mac_col) * pts
    tn = (2.0 * 2 * mac_sdf + 1 * 2 * mac_col) * pts
    clip = 2 * 17.6e9
    return mlp, nt, tn, clip


def placement_flops_per_step():
    """The 0.875 F_sdf of the sample-placement passes (coarse + 3 up-sampling rounds): executed by the fused value-chain
    kernel (avc::chain::k_sdf_chain) when it is on, by the NT tiles otherwise."""
    mac_sdf = 39 * 256 + 6 * 256 * 256 + 256 * 217 + 256 * 257
    return 0.875 * 2 * mac_sdf * N_RAYS * (REN_KW["n_samples"] + REN_KW["n_importance"])


def host_cores() -> int:
    """Usable host cores: the cgroup CPU quota when there is one (the GPU boxes expose 128 logical CPUs but
    grant a 16-CPU quota; 128 threads then run ~50x slower than 16), else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    return n


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1425.6), d.get("hbm_gbs", 6566.4), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_weights():
    """Seeded synthetic weights of the workload (product-side generators; no test / oracle code involved)."""
    sp, cp = WL.synth_states(SDF_KW, COL_KW, seed=0)
    clip_sd = WL.random_vit_state(seed=0)
    text = torch.randn(2, 512, generator=torch.Generator().manual_seed(5))
    return sp, cp, clip_sd, text


def build_world(device, engine):
    from avatarclip_b200.clip_vit import ClipImageTower
    sp, cp, clip_sd, text = synth_weights()
    sdf, col, var, ren = WL.build_networks(SDF_KW, COL_KW, REN_KW, sp, cp, VARIANCE, device, engine=engine, chunk=4096)
    tower = ClipImageTower(clip_sd, device=device)
    return sp, cp, clip_sd, text, ren, tower


def parity_view():
    """View 0 of the workload with the per-ray jitter the UNMODIFIED reference render draws under
    torch.manual_seed(PARITY_JITTER_SEED) (renderer.py:317-319), so both sides place samples from the same draw."""
    hv = WL.make_view(0, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(PARITY_JITTER_SEED)
        hv.jitter.copy_((torch.rand([N_RAYS, 1]) - 0.5).reshape(-1))
    return hv


class StdoutToStderr:
    """NCCL (NCCL_DEBUG=INFO/VERSION) and other native libraries print on fd 1; the contract is ONE JSON line on stdout.
    While active, fd 1 points at stderr (so those logs stay visible to the driver there); `emit` writes to the real
    stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


def kernel_key(name):
    """'void avc::tc::gemm_tc_nt_kernel<128, 3, ...>(...)' -> 'avc::tc::gemm_tc_nt_kernel';
    'void (anonymous namespace)::k_gemm16<EpiFc>(...)' -> 'k_gemm16'."""
    import re
    n = re.sub(r"^void\s+", "", name).replace("(anonymous namespace)::", "")
    m = re.match(r"[A-Za-z_][A-Za-z0-9_:]*", n)
    return m.group(0) if m else n


def count_my_launches(fn):
    """Kernels of libavc_b200.so launched by one call of fn (torch.profiler / CUPTI), by name."""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        mine, total, table = 0, 0, {}
        for ev in prof.events():
            if ev.device_type is not None and str(ev.device_type).endswith("CUDA") and ev.name:
                total += 1
                n = ev.name
                if "avc::" in n or "k_gemm16" in n or "(anonymous namespace)::k_" in n or n.startswith("k_"):
                    mine += 1
                    key = kernel_key(n)
                    t = table.setdefault(key, [0, 0.0])
                    t[0] += 1
                    t[1] += ev.device_time if hasattr(ev, "device_time") else getattr(ev, "cuda_time", 0.0)
        return mine, total, table
    except Exception as e:  # pragma: no cover
        return None, None, {"error": repr(e)}


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(tr, loss):
    """What one training step hands its caller, copied to the host: the loss, the CLIP cosines and image embeddings, the
    loss stage's scalars, every render output, the flat gradient and the flat parameters / Adam moments after the update."""
    arrays = {"loss": loss, "clip_cos": tr.cos, "clip_image_embedding": tr.emb, "loss_scalars": tr.scalars,
              "grad": tr.grad, "params": tr.fp.flat, "adam_exp_avg": tr.exp_avg, "adam_exp_avg_sq": tr.exp_avg_sq}
    arrays.update({"render_" + k: v for k, v in tr._out.items() if torch.is_tensor(v)})
    out = {}
    for k, v in arrays.items():
        v = v.detach().cpu()
        out[k] = v.double().numpy() if v.dtype == torch.float64 or not v.is_floating_point() else v.float().numpy()
    return out


def write_outputs(directory, arrays):
    """One DIR/<name>.npy per array (float32, or float64 where the value is not a float32 tensor)."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES} byte budget")
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def run_native(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    pg = None
    real_stdout = StdoutToStderr()      # native-library chatter (NCCL INFO) goes to stderr, the JSON line to the real stdout
    if world > 1:
        import torch.distributed as dist
        # NCCL_DEBUG is left as the caller set it (INFO when unset, so the communicator's rank count is on record)
        os.environ.setdefault("NCCL_DEBUG", os.environ.get("AVC_NCCL_DEBUG", "INFO"))
        dist.init_process_group("nccl", device_id=device)
        pg = dist.group.WORLD
    from avatarclip_b200.trainer import AppearanceTrainer, DeviceView
    make_view = WL.make_view
    sp, cp, clip_sd, text, ren, tower = build_world(device, args.engine)
    tr = AppearanceTrainer(ren, tower, text, lr=5e-4, process_group=pg, device=device)
    # ---------------- parity probe at the initial weights (compared with the reference in the cpu_baseline leg)
    probe = None
    if rank == 0 and not args.no_cpu_baseline:
        pv = parity_view()
        tr.forward_backward(DeviceView(pv, device))
        torch.cuda.synchronize()
        probe = {"view": pv, "color_fine": tr._out["color_fine"].detach().cpu().clone(),
                 "extra_color_fine": tr._out["extra_color_fine"].detach().cpu().clone(),
                 "weight_sum": tr._out["weight_sum"].detach().cpu().clone(),
                 "cos": tr.cos.detach().cpu().clone(), "loss": float(tr.loss_value())}
    K, Wm = args.steps, args.warmup
    n_views = 8
    views = [make_view(rank + world * i, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3, pin=True)
             for i in range(n_views)]
    dv = DeviceView(views[0], device)
    resident = [DeviceView(v, device) for v in views]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (value) + per-phase events for the roofline
    for i in range(Wm):
        tr.step(resident[i % n_views])
    barrier()
    # one extra step on EVERY rank (it contains the all-reduce); only rank 0 records it with CUPTI
    launches_per_step, total_launches, table = (None, None, {})
    # The profiled step runs with PLAIN launches of the tcgen05 NeuS kernels (AVC_TC_PDL=0, read per launch): under
    # programmatic dependent launch a kernel's CUPTI record starts when its first CTA becomes resident and includes the
    # wait for its predecessor, so durations overlap; the roofline wants the kernel's own duration.
    old_pdl = os.environ.get("AVC_TC_PDL")
    os.environ["AVC_TC_PDL"] = "0"
    if rank == 0:
        launches_per_step, total_launches, table = count_my_launches(lambda: tr.step(resident[0]))
    else:
        tr.step(resident[0])
    if old_pdl is None:
        os.environ.pop("AVC_TC_PDL", None)
    else:
        os.environ["AVC_TC_PDL"] = old_pdl
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    use_graph = bool(args.graph)
    if use_graph:
        # the whole step as one CUDA graph on the static view `dv`; each step refreshes dv with ONE copy
        dv.copy_from(resident[0])
        tr.capture(dv)
        for i in range(2):
            dv.copy_from(resident[i % n_views])
            tr.replay(dv)
        barrier()

    def one_step(i):
        if use_graph:
            dv.copy_from(resident[i % n_views])      # D2D, inputs resident in HBM
            return tr.replay(dv)
        return tr.step(resident[i % n_views])

    ev[0].record()
    for i in range(K):
        loss = one_step(i)
    ev[1].record()
    barrier()
    ms_value = ev[0].elapsed_time(ev[1])
    # the steps below (render-only timing, phases, end to end) train on: snapshot the timed path's last step now
    dumped = step_outputs(tr, loss) if args.dump_outputs and rank == 0 else None
    clocks = sampler.stop() if rank == 0 else None

    # render-only share (events around the two render calls) for the roofline of the MLP contractions
    from avatarclip_b200 import renderer as R
    tot_render = 0.0
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for i in range(min(K, 5)):
        d = resident[i % n_views]
        e[0].record()
        out, ws, chunk = R.render_forward_raw(ren, d.rays_o, d.rays_d, d.near, d.far, d.jitter, None, 0, 1.0, None,
                                              keep_ws=False, out=tr._out)
        e[1].record()
        cot = {k: torch.ones_like(out[k]) for k in ("color_fine", "extra_color_fine", "weights", "gradients")}
        e[2].record()
        R.render_backward_raw(ren, d.rays_o, d.rays_d, None, 0, 1.0, out, ws, chunk, cot, grad=tr.grad)
        e[3].record()
        torch.cuda.synchronize()
        tot_render += e[0].elapsed_time(e[1]) + e[2].elapsed_time(e[3])
    ms_render = tot_render / min(K, 5)

    # per-phase device times (CUDA events between the C-ABI calls), averaged over a few extra steps
    phases = {}
    for i in range(5):
        tr.phase_events = []
        tr.step(resident[i % n_views])
        torch.cuda.synchronize()
        evs = tr.phase_events
        for (n0, e0), (n1, e1) in zip(evs[:-1], evs[1:]):
            phases[n1] = phases.get(n1, 0.0) + e0.elapsed_time(e1) / 5.0
    tr.phase_events = None

    # ---------------- end-to-end timing: pinned-host inputs copied every step, loss read back every step
    barrier()
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    # The loss of step i is copied to pinned host memory on the stream right after step i and read by the host
    # while step i+1 runs (the reference logs its loss the same lagged way only every report_freq steps); every
    # step's loss is read inside the timed region, the last one before the closing synchronise.
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    done = [torch.cuda.Event() for _ in range(K)]
    ev2[0].record()
    last = 0.0
    for i in range(K):
        dv.upload(views[i % n_views])                # one H2D copy of the packed, pinned view
        loss = tr.replay(dv) if use_graph else tr.step(dv)
        loss_host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
        done[i].record()
        if i > 0:
            done[i - 1].synchronize()
            last = float(loss_host[i - 1])
    done[K - 1].synchronize()
    last = float(loss_host[K - 1])
    ev2[1].record()
    barrier()
    ms_e2e = ev2[0].elapsed_time(ev2[1])

    t = torch.tensor([ms_value, ms_e2e], device=device)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_value, ms_e2e = t.tolist()

    if rank == 0:
        mlp_flops, nt_flops, tn_flops, clip_flops = algorithmic_flops_per_step()
        peak_tf, peak_hbm, peak_src = peaks()
        achieved_step = mlp_flops / (ms_render * 1e-3) / 1e12
        # The CLIP tower's kernels are chained with programmatic dependent launch: each starts early and its CUPTI
        # duration includes the time it spends in griddepcontrol.wait for its predecessor, so those durations overlap
        # and do not add up (phases_ms.clip_* are the true times).  The dominant kernel is picked among the rest.
        plain = {k: v for k, v in table.items() if isinstance(v, list) and k.startswith("avc::")}
        dom = max(plain.items(), key=lambda kv: kv[1][1])[0] if plain else None
        # dominant kernel: algorithmic FLOP its launches execute per step / the sum of their device durations in the
        # profiled step (CUPTI kernel records taken live in this process, not under ncu)
        kern_us = {k: v for k, v in table.items() if isinstance(v, list)}
        chain_on = "avc::chain::k_sdf_chain" in kern_us
        if chain_on:
            nt_flops -= placement_flops_per_step()
        dom_flops = {"avc::tc::gemm_tc_nt_kernel": nt_flops, "avc::chain::k_sdf_chain": placement_flops_per_step(), "avc::tc::gemm_tc_tn_kernel": tn_flops,
                     "avc::gemm_nt_kernel": nt_flops, "avc::gemm_tn_kernel": tn_flops}.get(dom)
        if dom_flops is not None and dom in kern_us and kern_us[dom][1] > 0:
            n_launch, dom_us = kern_us[dom]
            achieved = dom_flops / (dom_us * 1e-6) / 1e12
            per_launch = {"launches_per_step": n_launch, "avg_launch_us": dom_us / n_launch,
                          "algorithmic_gflop_per_launch": dom_flops / n_launch / 1e9}
        else:
            achieved, per_launch = achieved_step, None
        line = {
            "metric": METRIC, "value": world * K / (ms_value * 1e-3), "unit": "steps/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": ms_value / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.engine == 0 else "bf16x3(split)->f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "views_per_step": world, "engine": "fp32 FFMA tiles" if args.engine == 0 else "tcgen05 split",
                       "l2": "per-step working set (activation stash ~2.4 GB) >> 126 MB L2; no flush needed",
                       "parallelism": f"view-sharded dp{world}" if world > 1 else "single",
                       "launch": ("one CUDA graph per step" + ((" (NCCL all-reduce + Adam captured inside)" if tr._graph_has_adam
                                                                 else " + all-reduce + Adam after it") if world > 1 else ""))
                                 if use_graph else "eager C-ABI calls"},
            "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "steps/s",
                    "h2d_bytes_per_step": views[0].h2d_bytes(), "d2h_bytes_per_step": 4},
            "gpu_launches": None if launches_per_step is None else launches_per_step * K,
            "gpu_launches_per_step": launches_per_step,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved / peak_tf,
                         "traffic": TRAFFIC_PER_LAUNCH.get(dom),
                         "per_launch": per_launch,
                         "scope": "algorithmic FLOP executed by the dominant kernel's launches in one step (SURVEY 8d "
                                  "split: NT tiles 4.875 F_sdf + 2 F_col per point -- 4.0 F_sdf when the fused value-chain "
                                  "kernel runs the 0.875 F_sdf of the placement passes --, TN tiles 2 F_sdf + F_col) / sum of "
                                  "their device durations (CUPTI, live, taken on a step with plain launches: under programmatic dependent launch a record includes the wait for the predecessor); peak = " + peak_src + "; the kernel runs 3 "
                                  "bf16 MMAs per product (two-term split), so its ceiling is peak/3",
                         "hbm_view": (lambda b, us: {"designed_bytes_per_step": b, "kernel_us_per_step": us,
                                                     "achieved_GBps": b / (us * 1e-6) / 1e9 if us else None,
                                                     "peak_GBps": peak_hbm,
                                                     "frac": (b / (us * 1e-6) / 1e9 / peak_hbm) if us else None,
                                                     "note": "the layers are not fused, so the NT launches are bound by "
                                                             "the activation traffic they move by design (operands in, "
                                                             "stash + split out), not by the tensor pipe"})(
                             nt_designed_bytes_per_step(), kern_us.get("avc::tc::gemm_tc_nt_kernel", [0, 0.0])[1]),
                         "fused_chain": ({"kernel": "avc::chain::k_sdf_chain", "launches_per_step": kern_us["avc::chain::k_sdf_chain"][0],
                                          "us_per_step": kern_us["avc::chain::k_sdf_chain"][1],
                                          "achieved": placement_flops_per_step() / (kern_us["avc::chain::k_sdf_chain"][1] * 1e-6) / 1e12,
                                          "frac": placement_flops_per_step() / (kern_us["avc::chain::k_sdf_chain"][1] * 1e-6) / 1e12 / peak_tf,
                                          "hbm_bytes_per_point": 164} if chain_on else None),
                         "step_level": {"achieved": achieved_step, "frac": achieved_step / peak_tf,
                                        "ms_render_fwd_bwd": ms_render,
                                        "note": "all MLP FLOP/step (0.577 T) / CUDA-event time of render fwd+bwd"},
                         "kernel_time_us_per_step": {k: round(v[1], 1) for k, v in
                                                     sorted(((k, v) for k, v in kern_us.items() if k.startswith("avc::")),
                                                            key=lambda kv: -kv[1][1])[:8]}},
            "last_loss": last,
            "phases_ms": {k: round(v, 4) for k, v in phases.items()},
        }
        clip_ms = phases.get("clip_fwd", 0.0) + phases.get("clip_bwd", 0.0)
        if clip_ms > 0:
            gbps = 2 * CLIP_WEIGHT_BYTES_PER_PASS / (clip_ms * 1e-3) / 1e9
            line["roofline_clip"] = {"bound": "hbm", "achieved": gbps, "peak": peak_hbm, "unit": "GB/s",
                                     "frac": gbps / peak_hbm, "ms_fwd_bwd": clip_ms,
                                     "tensor_tflops": clip_flops / (clip_ms * 1e-3) / 1e12,
                                     "scope": "CLIP ViT-B/32 on 2 canvases: fp16 weight stream of the forward and of the "
                                              "input-gradient backward (2 x 175.7 MB) / CUDA-event time of the two calls"}
        if not args.no_cpu_baseline:
            cb, parity = cpu_baseline(sp, cp, clip_sd, text, probe, budget_s=args.cpu_budget_s)
            line["cpu_baseline"] = cb
            line["parity"] = parity
            if args.ref_gpu:
                line["ref_gpu"] = reference_gpu(sp, cp, clip_sd, text, device, steps=max(5, min(K, 20)))
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
            line["dump_outputs"] = {"dir": args.dump_outputs, "arrays": sorted(dumped),
                                    "step": "last timed step (after warm-up, the profiled step and the timed steps)"}
        real_stdout.emit(json.dumps(line))
    if world > 1:
        tr.release_graph()          # the graph may hold the NCCL all-reduce: it has to go before the communicator
        del tr
        import gc
        gc.collect()
        torch.cuda.synchronize()
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# Reference arms.  The ONLY code in this file that touches oracle/: the checker / timed baseline, never the product.
# ------------------------------------------------------------------------------------------------------------------
def reference_trainer(sp, cp, clip_sd, text, device="cpu", clip_half=False):
    """The reference's unmodified renderer (oracle/_ref, staged by oracle/make_ref.py) inside the restated step;
    falls back to the oracle port when the staged files are absent (kind says which)."""
    from oracle import make_ref
    if make_ref.available():
        from oracle.ref_step import ReferenceTrainer
        return ReferenceTrainer(SDF_KW, COL_KW, REN_KW, sp, cp, VARIANCE, clip_sd, text, lr=5e-4, device=device,
                                clip_half=clip_half), "reference"
    if device != "cpu":
        raise RuntimeError("oracle/_ref is not staged: no reference GPU arm")
    from oracle import neus
    from oracle.train_step import OracleTrainer
    sconf = neus.SDFConf(**{k: (tuple(v) if k == "skip_in" else v) for k, v in SDF_KW.items()})
    return OracleTrainer(sconf, neus.ColorConf(**COL_KW), neus.RenderConf(**REN_KW), sp, cp, VARIANCE, clip_sd, text,
                         lr=5e-4), "port"


def cpu_baseline(sp, cp, clip_sd, text, probe, budget_s=20.0):
    """The reference step on this box's host cores on the FULL workload (512 rays), as many steps as fit in
    ~budget_s (>= 2) after one warm-up step; and the parity of the native arm's probe against the reference's forward
    on the same view, weights and jitter draw."""
    torch.set_num_threads(host_cores())
    ref, kind = reference_trainer(sp, cp, clip_sd, text)
    pv = probe["view"]
    # ---- parity (forward at the initial weights)
    t0 = time.perf_counter()
    if kind == "reference":
        total, aux = ref.loss(pv, jitter_seed=PARITY_JITTER_SEED)
    else:
        total, aux = ref.loss(pv)
    t_fwd = time.perf_counter() - t0
    o = aux["out"]
    rel = lambda a, b: float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-12))
    ec_ref, c_ref = o["extra_color_fine"].detach(), o["color_fine"].detach()
    dray = torch.maximum((probe["extra_color_fine"] - ec_ref).abs().max(dim=1)[0],
                         (probe["color_fine"] - c_ref).abs().max(dim=1)[0])
    cl_ref = float((1.0 - aux["cos"]).sum())
    cl_nat = float((1.0 - probe["cos"]).sum())
    parity = {"against": kind + " renderer + restated loss stage + CLIP stand-in (fp32, CPU), same view / weights / jitter",
              "rays": int(ec_ref.shape[0]),
              "rgb_rel": max(rel(probe["extra_color_fine"], ec_ref), rel(probe["color_fine"], c_ref)),
              "frac_rays_1e-3": float((dray < 1e-3).float().mean()),
              "median_ray_abs": float(dray.median()),
              "weight_sum_rel": rel(probe["weight_sum"], o["weight_sum"].detach()),
              "clip_loss_rel": abs(cl_nat - cl_ref) / abs(cl_ref),
              "total_loss_rel": abs(probe["loss"] - float(total)) / abs(float(total)),
              "cos_native": [float(x) for x in probe["cos"]], "cos_reference": [float(x) for x in aux["cos"]]}
    del total, aux, o
    # ---- timing
    views = [WL.make_view(i, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3) for i in range(4)]
    t0 = time.perf_counter()
    ref.step(views[0])
    t_warm = time.perf_counter() - t0
    n = max(2, min(12, int(budget_s / max(t_warm, 1e-3))))
    t0 = time.perf_counter()
    for i in range(n):
        ref.step(views[(i + 1) % 4])
    t = (time.perf_counter() - t0) / n
    cb = {"value": 1.0 / t, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": kind,
          "sample": f"{n} full steps (512 rays x 128 samples, CLIP x2, backward, Adam) after 1 warm-up; "
                    f"{t:.2f} s/step; forward alone {t_fwd:.2f} s"}
    return cb, parity


def reference_gpu(sp, cp, clip_sd, text, device, steps=10):
    """The reference's own renderer on THIS GPU the way the reference runs it (main.py:948 default CUDA tensors, fp32
    eager PyTorch, CLIP stand-in in fp16 like clip.load): the 'reference single-GPU PyTorch' denominator of north_star."""
    try:
        ref, kind = reference_trainer(sp, cp, clip_sd, text, device=str(device), clip_half=True)
        prev_tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        views = [WL.make_view(i, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3) for i in range(4)]
        for i in range(3):
            ref.step(views[i % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for i in range(steps):
            last, _ = ref.step(views[i % 4])
        e1.record()
        torch.cuda.synchronize()
        torch.backends.cuda.matmul.allow_tf32 = prev_tf32
        ms = e0.elapsed_time(e1) / steps
        return {"value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "steps": steps, "last_loss": float(last),
                "what": "UNMODIFIED reference renderer.py/fields.py/embedder.py (oracle/_ref) under "
                        "torch.set_default_tensor_type('torch.cuda.FloatTensor') as main.py:948, fp32 eager, "
                        "allow_tf32=False; restated loss stage; CLIP stand-in fp16; torch.optim.Adam; same workload"}
    except Exception as e:  # pragma: no cover
        torch.set_default_tensor_type("torch.FloatTensor")
        return {"unavailable": repr(e)[:200]}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores -- its unmodified
    renderer files (oracle/_ref) inside the restated step -- on the FULL workload of the native arm, no extrapolation."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    torch.set_num_threads(host_cores())
    sp, cp, clip_sd, text = synth_weights()
    ref, kind = reference_trainer(sp, cp, clip_sd, text)
    views = [WL.make_view(i, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3) for i in range(4)]
    for i in range(args.warmup):
        ref.step(views[i % 4])
    t0 = time.perf_counter()
    for i in range(args.steps):
        ref.step(views[i % 4])
    tot = time.perf_counter() - t0
    val = args.steps / tot
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the native arm's workload string verbatim + what differs in THIS arm (rank 0 alone runs it: one view per step)
            "config": {"workload": WORKLOAD, "views_per_step": 1, "engine": "reference algorithm, torch fp32 eager",
                       "parallelism": "host cores of rank 0", "launch": "unmodified reference renderer (oracle/_ref) inside "
                       "the restated step; full ray count, no extrapolation" if kind == "reference" else
                       "oracle port of the reference renderer; full ray count, no extrapolation"},
            "cpu_baseline": {"value": val, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": f"{args.steps} full steps (512 rays), unmodified reference renderer"
                                       if kind == "reference" else f"{args.steps} full steps (512 rays), oracle port"},
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# The other BASELINE.json configurations (parity-test cases of the tier, benchable on request): --config 2 | 3 | 4
# ------------------------------------------------------------------------------------------------------------------
def run_other_config(args):
    """configs[2]: full 224 x 224 views (50 176 rays each, chunked forward + recompute backward), `--batch-views B` views
    accumulated per optimiser step and sharded over the ranks (B = world: weak scaling, one view per GPU; B = 8 fixed:
    strong scaling of an 8-view batch).  configs[3]: configs[1] + SMPL linear-blend skinning of the 6890-vertex template
    inside every step.  configs[4]: the real train_clip loop (Runner, shipped-size nets, per-step camera draw + template
    raster + silhouette rays on the device, ~max_ray_num rays), throughput + final CLIP cosine."""
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    real_stdout = StdoutToStderr()
    pg = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", os.environ.get("AVC_NCCL_DEBUG", "INFO"))
        dist.init_process_group("nccl", device_id=device)
        pg = dist.group.WORLD
    from avatarclip_b200.trainer import AppearanceTrainer, DeviceView
    K, Wm = args.steps, args.warmup
    cfg = args.config

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    extra = {}
    if cfg in (2, 3):
        sp, cp, clip_sd, text, ren, tower = build_world(device, args.engine)
        tr = AppearanceTrainer(ren, tower, text, lr=5e-4, process_group=pg, device=device)
        if cfg == 2:
            B = args.batch_views if args.batch_views > 0 else world
            if B % world:
                raise SystemExit("--batch-views must be a multiple of the number of ranks")
            per_rank = B // world
            n_rays = CANVAS * CANVAS
            views = [DeviceView(WL.make_view(rank * per_rank + i, n_rays=n_rays, H=CANVAS, W=CANVAS, seed=0, bg_choice=3,
                                             radius=1.5), device) for i in range(per_rank)]

            def step(i):
                acc = None
                for v in views:                                  # gradient accumulation over this rank's views
                    g = tr.forward_backward(v)
                    acc = g.clone() if (acc is None and per_rank > 1) else (g if acc is None else acc.add_(g))
                if acc is not tr.grad:
                    tr.grad.copy_(acc)
                tr.optimizer_step()
            units = B
            workload = (f"BASELINE configs[2]: {B} views x 224x224 = {n_rays} rays each x (64+64) samples per optimiser step, "
                        f"8x256 SDF + 4x256 colour, CLIP loss per view, chunked render (4096-ray chunks, backward recompute); "
                        f"{per_rank} view(s) per GPU, gradients accumulated then all-reduced")
            scaling = "strong" if args.batch_views > 0 else "weak"
            metric, unit = "appearance-optim views/sec (224x224 full views, CLIP loss)", "views/s"
        else:
            from avatarclip_b200.lbs import my_lbs
            smpl = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in WL.synthetic_smpl().items()}
            views = [DeviceView(WL.make_view(rank + world * i, n_rays=N_RAYS, H=CANVAS, W=CANVAS, seed=0, bg_choice=3), device)
                     for i in range(8)]

            def step(i):
                verts, _ = my_lbs(smpl["v_shaped"], smpl["pose"], None, None, smpl["posedirs"], smpl["J_regressor"],
                                  smpl["parents"], smpl["lbs_weights"], pose2rot=True)
                extra["verts_checksum"] = verts
                tr.step(views[i % 8])
            units = world
            workload = ("BASELINE configs[3]: configs[1] step + avc_lbs_fwd (my_lbs, 6890-vertex template, 24 joints, "
                        "synthetic SMPL tensors) inside every step; 1 view per GPU per step")
            scaling, metric, unit = "weak", METRIC + " + LBS per step", "steps/s"
    else:
        import tempfile
        from avatarclip_b200.runner import Runner
        tmp = tempfile.mkdtemp(prefix="avc_cfg4_")
        conf = f"""
general {{ base_exp_dir = {tmp}/exp }}
dataset {{ data_dir = {tmp}/none }}
train {{ learning_rate = 5e-4
  learning_rate_alpha = 0.05
  end_iter = 100000
  batch_size = 512
  warm_up_end = 500
  anneal_end = 0
  save_freq = 100000
  val_freq = 100000
  val_mesh_freq = 100000
  report_freq = 100000
  igr_weight = 0.1
  mask_weight = 0.5
  clip_weight = 1.0
  add_no_texture = True
  texture_cast_light = True
  use_face_prompt = True
  use_back_prompt = True
  use_silhouettes = True
  seed = 1000 }}
clip {{ prompt = a 3D rendering of the Iron Man in unreal engine }}
model {{
  sdf_network {{ d_out = 257, d_in = 3, d_hidden = 256, n_layers = 4, skip_in = [4], multires = 6, bias = 0.5, scale = 1.0, geometric_init = True, weight_norm = True }}
  variance_network {{ init_val = 0.3 }}
  rendering_network {{ d_feature = 256, mode = no_view_dir, d_in = 6, d_out = 3, d_hidden = 256, n_layers = 2, weight_norm = True, multires_view = 0, squeeze_out = True, extra_color = True }}
  neus_renderer {{ n_samples = 32, n_importance = 32, n_outside = 0, up_sample_steps = 4, perturb = 1.0, extra_color = True }}
}}"""
        cpath = os.path.join(tmp, "ironman_like.conf")
        open(cpath, "w").write(conf)
        r = Runner(cpath, mode="train_clip", case="smpl", device=str(device), engine=args.engine)
        g = torch.Generator().manual_seed(5)
        r.init_clip(WL.random_vit_state(seed=0), torch.randn(1, 512, generator=g), torch.randn(1, 512, generator=g),
                    torch.randn(1, 512, generator=g))
        v, f = WL.synthetic_body_mesh()
        r.init_smpl(v, f)
        r.set_process_group(pg)
        state = {"done": 0}

        def step(i):
            pass
        units = world
        workload = ("BASELINE configs[4]-like: Runner.train_clip real loop, shipped-size nets (4x256 + 2x256, 32+32 samples), "
                    "max_ray_num 12544 (~11-12.5 k silhouette rays / step), per-step camera draw + template raster + "
                    "dilation + canvas + rays on the device with one-step lookahead, face/back prompts, bg augmentation; "
                    "synthetic body mesh, seeded random CLIP weights (stand-ins for the licence-gated assets)")
        scaling, metric, unit = "weak", "appearance-optim steps/sec (real train_clip loop, ~12 k rays x 64 samples, CLIP loss)", "steps/s"

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    if cfg == 4:
        r.train_clip(max_steps=Wm, log=lambda m: None, validate=False)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ev[0].record()
        r.train_clip(max_steps=K, log=lambda m: None, validate=False)
        ev[1].record()
        barrier()
        extra["final_clip_cosine"] = [float(x) for x in r.trainer.cos]
        extra["rays_last_step"] = int(r.trainer._out["weights"].shape[0])
    else:
        for i in range(Wm):
            step(i)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ev[0].record()
        for i in range(K):
            step(i)
        ev[1].record()
        barrier()
    ms = ev[0].elapsed_time(ev[1])
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=device)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t[0])
    if rank == 0:
        line = {"metric": metric, "value": units * K / (ms * 1e-3), "unit": unit, "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "f32" if args.engine == 0 else "bf16x3(split)->f32", "data": "synthetic",
                "config": {"workload": workload, "baseline_config": cfg, "parallelism": f"view-sharded dp{world}" if world > 1 else "single",
                           "launch": "eager C-ABI calls", "l2": "working set >> 126 MB L2"},
                "clocks": clocks, "last_loss": float(tr.loss_value()) if cfg in (2, 3) else float(r.trainer.loss_value())}
        for k, v in extra.items():
            if not torch.is_tensor(v):
                line[k] = v
        real_stdout.emit(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--engine", type=int, default=int(os.environ.get("AVC_ENGINE", "1")),
                    help="MLP contraction engine: 1 = tcgen05 split-bf16 tiles (default), 0 = fp32 FFMA tiles")
    ap.add_argument("--graph", type=int, default=int(os.environ.get("AVC_GRAPH", "1")),
                    help="1: replay the step as one captured CUDA graph (default); 0: eager C-ABI calls")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4],
                    help="BASELINE.json configs index (default 1 = the headline config; 2, 3, 4: see run_other_config)")
    ap.add_argument("--batch-views", type=int, default=0,
                    help="--config 2: views per optimiser step over ALL ranks (0: one per rank = weak scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true",
                    help="skip the cpu_baseline / parity / ref_gpu legs (kernel experiments)")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="CPU seconds the cpu_baseline leg may spend on steps")
    ap.add_argument("--ref-gpu", type=int, default=1, help="1: also time the unmodified reference renderer on this GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, CLIP cosines, render outputs, gradient, parameters "
                         "after the update) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.config != 1):
        ap.error("--dump-outputs is available for the native arm of configs[1]")
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback")
        if args.config != 1:
            run_other_config(args)
        else:
            run_native(args)


if __name__ == "__main__":
    main()
