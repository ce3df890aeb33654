"""Shared helpers for the NeuS parity tests: build the product modules from oracle / golden weights,
run the CUDA path and the CPU oracle on identical inputs and report errors."""
from __future__ import annotations

import math
import os
from typing import Dict, Optional

import torch

from oracle import neus

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

COT_KEYS = ["color_fine", "extra_color_fine", "s_val", "cdf_fine", "weight_sum", "weight_max", "gradients",
            "weights", "gradient_error"]


def log_parity(name: str, rec: dict):
    """Append one measured-parity record to gpurun_out/r2_parity.jsonl (merged into profiles/ by tools/collect_parity.py):
    the tests assert bars, this file keeps the numbers actually measured on the GPU box."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = os.path.join(root, "gpurun_out")
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "r2_parity.jsonl"), "a") as f:
            f.write(json.dumps(dict(test=name, **rec)) + "\n")
    except OSError:
        pass


def sm_count() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def nt_tiles_per_cta(M: int, N: int) -> int:
    """Row tiles the first CTA of a tcgen05 NT launch walks (launch_gemm_tc_nt_bn's grid: min(tiles, SMs) persistent
    CTAs, a whole number per column tile; BN = 64 for N <= 64, else 128)."""
    BN = 64 if N <= 64 else 128
    tiles_n, tiles_m = -(-N // BN), -(-M // 128)
    m_stride = min(tiles_m * tiles_n, sm_count()) // tiles_n
    return -(-tiles_m // m_stride)


def chain_tiles_per_cta(P: int) -> int:
    """128-point tiles the first CTA of the fused value chain walks (min(tiles, SMs) persistent CTAs)."""
    tiles = -(-P // 128)
    return -(-tiles // min(tiles, sm_count()))


def flat_rel_l2(got: Dict[str, torch.Tensor], ref: Dict[str, torch.Tensor]) -> float:
    """rel-L2 error of the concatenated parameter gradient."""
    num = sum((got[k].double().cpu() - ref[k].double().cpu()).pow(2).sum().item() for k in ref)
    den = sum(ref[k].double().pow(2).sum().item() for k in ref)
    return (num / max(den, 1e-300)) ** 0.5


def confs_from_kw(sdf_kw, col_kw, ren_kw):
    sconf = neus.SDFConf(**{k: (tuple(v) if k == "skip_in" else v) for k, v in sdf_kw.items()})
    return sconf, neus.ColorConf(**col_kw), neus.RenderConf(**ren_kw)


def build_product(sdf_kw, col_kw, ren_kw, sdf_state, col_state, variance, device, engine=0, chunk=4096,
                  **renderer_kw):
    """``renderer_kw``: further NeuSRenderer options (color_products, wgrad_products)."""
    import avatarclip_b200 as ab
    sdf = ab.SDFNetwork(**sdf_kw)
    col = ab.RenderingNetwork(**col_kw)
    var = ab.SingleVarianceNetwork(float(variance))
    sdf.load_state_dict(sdf_state)
    col.load_state_dict(col_state, strict=False)
    sdf, col, var = sdf.to(device), col.to(device), var.to(device)
    ren = ab.NeuSRenderer(None, sdf, var, col, engine=engine, max_rays_per_chunk=chunk, **ren_kw, **renderer_kw)
    return sdf, col, var, ren


def rel_to_max(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / (b.abs().max().item() + 1e-12)


def make_rays(R, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    d = torch.randn(R, 3, generator=g, dtype=dtype) * 0.25 + torch.tensor([0.0, 0.0, -1.0], dtype=dtype)
    d = d / d.norm(dim=-1, keepdim=True)
    o = torch.tensor([0.0, 0.0, 1.8], dtype=dtype) + 0.05 * torch.randn(R, 3, generator=g, dtype=dtype)
    near, far = neus.near_far_from_sphere(o, d)
    jit = torch.rand(R, 1, generator=g, dtype=dtype) - 0.5
    return o, d, near, far, jit


def cotangents(out: Dict[str, torch.Tensor], seed=7):
    g = torch.Generator().manual_seed(seed)
    c = {}
    for k in COT_KEYS:
        c[k] = torch.randn(out[k].shape, generator=g) * (0.05 if k == "gradients" else 1.0)
    return c


def oracle_run(sconf, cconf, rconf, sdf_state, col_state, variance, o, d, near, far, jit, bg, anneal, cot=None,
               z_vals=None, dtype=torch.float32):
    sp = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in sdf_state.items()}
    cp = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in col_state.items()}
    var = torch.as_tensor(variance).detach().to(dtype).clone().requires_grad_(True)
    cv = lambda t: None if t is None else t.to(dtype)
    out = neus.render(sp, cp, var, sconf, cconf, rconf, cv(o), cv(d), cv(near), cv(far), jitter=cv(jit),
                      background_rgb=cv(bg), cos_anneal_ratio=anneal, z_vals=cv(z_vals))
    grads = None
    if cot is not None:
        loss = sum((out[k] * cot[k].to(dtype)).sum() for k in cot)
        names = [("sdf." + k, v) for k, v in sp.items()] + [("col." + k, v) for k, v in cp.items()] + [("var.variance", var)]
        gs = torch.autograd.grad(loss, [v for _, v in names], allow_unused=True)
        grads = {k: (torch.zeros_like(v) if g is None else g) for (k, v), g in zip(names, gs)}
    return out, grads


def product_run(ren, sdf, col, var, o, d, near, far, jit, bg, anneal, cot=None, z_vals=None, device="cuda"):
    dev = torch.device(device)
    to = lambda t: None if t is None else t.to(dev)
    for m in (sdf, col, var):
        for p in m.parameters():
            p.grad = None
    out = ren.render(to(o), to(d), to(near), to(far), perturb_overwrite=(1 if jit is not None else 0),
                     background_rgb=to(bg), cos_anneal_ratio=anneal, jitter=to(jit), z_vals=to(z_vals))
    grads = None
    if cot is not None:
        loss = sum((out[k] * cot[k].to(dev)).sum() for k in cot)
        loss.backward()
        grads = {}
        for pre, m in (("sdf.", sdf), ("col.", col), ("var.", var)):
            for k, p in m.named_parameters():
                grads[pre + k] = p.grad.detach().cpu() if p.grad is not None else torch.zeros_like(p).cpu()
    return {k: v.detach().cpu() for k, v in out.items()}, grads


CASES = {
    # name: (sdf_kw, col_kw, ren_kw, R)
    "tiny": (dict(d_in=3, d_out=33, d_hidden=32 + 16, n_layers=3, skip_in=[2], multires=6, bias=0.5, scale=1.0,
                  geometric_init=True, weight_norm=True),
             dict(d_feature=32, mode="no_view_dir", d_in=6, d_out=3, d_hidden=40, n_layers=2, weight_norm=True,
                  multires_view=0, squeeze_out=True, extra_color=True),
             dict(n_samples=16, n_importance=16, n_outside=0, up_sample_steps=4, perturb=1.0, extra_color=True), 40),
    "skiplast": (dict(d_in=3, d_out=65, d_hidden=64, n_layers=4, skip_in=[4], multires=6, bias=0.5, scale=1.0,
                      geometric_init=True, weight_norm=True),
                 dict(d_feature=64, mode="no_view_dir", d_in=6, d_out=3, d_hidden=64, n_layers=1, weight_norm=True,
                      multires_view=0, squeeze_out=True, extra_color=True),
                 dict(n_samples=24, n_importance=16, n_outside=0, up_sample_steps=2, perturb=1.0, extra_color=True), 70),
    "b2": (dict(d_in=3, d_out=257, d_hidden=256, n_layers=8, skip_in=[4], multires=6, bias=0.5, scale=1.0,
                geometric_init=True, weight_norm=True),
           dict(d_feature=256, mode="no_view_dir", d_in=6, d_out=3, d_hidden=256, n_layers=4, weight_norm=True,
                multires_view=0, squeeze_out=True, extra_color=True),
           dict(n_samples=64, n_importance=64, n_outside=0, up_sample_steps=4, perturb=1.0, extra_color=True), 48),
    "shipped": (dict(d_in=3, d_out=257, d_hidden=256, n_layers=4, skip_in=[4], multires=6, bias=0.5, scale=1.0,
                     geometric_init=True, weight_norm=True),
                dict(d_feature=256, mode="no_view_dir", d_in=6, d_out=3, d_hidden=256, n_layers=2, weight_norm=True,
                     multires_view=0, squeeze_out=True, extra_color=True),
                dict(n_samples=32, n_importance=32, n_outside=0, up_sample_steps=4, perturb=1.0, extra_color=True), 64),
}


def synth_state(sdf_kw, col_kw, seed=0, tame=True):
    """Seeded weights from the oracle's restated initialisers.  ``tame`` nudges the geometric init so the
    field stays SDF-like when the skip concat feeds the LAST linear (see DESIGN.md, 'parity definition')."""
    sconf, cconf, _ = confs_from_kw(sdf_kw, col_kw, dict())
    g = torch.Generator().manual_seed(seed)
    sp = neus.init_sdf_params(sconf, g)
    cp = neus.init_color_params(cconf, g)
    if tame:
        L = sconf.n_lin - 1
        if L in sconf.skip_in:
            with torch.no_grad():   # the last linear reads raw sin/cos features with weight sqrt(pi)/sqrt(K): damp them
                sp[f"lin{L}.weight_v"][:, -(sconf.d_enc - 3):] *= 0.02
                sp[f"lin{L}.weight_g"] = sp[f"lin{L}.weight_v"].norm(dim=1, keepdim=True)
        for k in sp:
            if k.endswith("weight_v"):
                sp[k] = sp[k] + 0.01 * torch.randn(sp[k].shape, generator=g)
    return sp, cp


def oracle_case(name: str, seed=0, bg_kind="ray", anneal=1.0, R: Optional[int] = None,
                oracle_dtype=torch.float32) -> dict:
    """Inputs of a synthetic case and the oracle's results on them: the full pipeline (sample placement) in fp32, as
    the reference runs it, then the fine pass and its backward on the oracle's own depths in ``oracle_dtype``."""
    sdf_kw, col_kw, ren_kw, Rdef = CASES[name]
    R = R or Rdef
    sconf, cconf, rconf = confs_from_kw(sdf_kw, col_kw, ren_kw)
    sp, cp = synth_state(sdf_kw, col_kw, seed)
    variance = 0.3
    o, d, near, far, jit = make_rays(R, seed + 1)
    g = torch.Generator().manual_seed(seed + 2)
    bg = {"none": None, "white": torch.ones(1, 3), "ray": torch.rand(R, 1, generator=g)}[bg_kind]
    rays = (o, d, near, far, jit, bg, anneal)
    oout, _ = oracle_run(sconf, cconf, rconf, sp, cp, variance, *rays)
    z = oout["z_vals"].detach()
    cot = cotangents(oout)
    oout2, ograds = oracle_run(sconf, cconf, rconf, sp, cp, variance, *rays, cot=cot, z_vals=z, dtype=oracle_dtype)
    return {"name": name, "R": R, "sp": sp, "cp": cp, "variance": variance, "rays": rays, "placement": oout, "z": z,
            "cot": cot, "fine": oout2, "grads": ograds, "oracle_dtype": str(oracle_dtype).replace("torch.", "")}


def run_case_gpu_vs_oracle(name: str, device="cuda", engine=0, seed=0, bg_kind="ray", anneal=1.0, chunk=4096,
                           R: Optional[int] = None, oracle_dtype=torch.float32, oracle: Optional[dict] = None,
                           **renderer_kw):
    """Full comparison on a synthetic case.  Returns a report dict with worst errors and 'ok'.  ``oracle``: the result
    of oracle_case for the same case (computed here when None; the other case arguments are then ignored).
    ``renderer_kw``: further NeuSRenderer options."""
    if oracle is None:
        oracle = oracle_case(name, seed, bg_kind, anneal, R, oracle_dtype)
    sdf_kw, col_kw, ren_kw, _ = CASES[oracle["name"]]
    R = oracle["R"]
    sp, cp, variance, rays = oracle["sp"], oracle["cp"], oracle["variance"], oracle["rays"]
    sdf, col, var, ren = build_product(sdf_kw, col_kw, ren_kw, sp, cp, variance, device, engine=engine, chunk=chunk,
                                       **renderer_kw)

    # (1) placement
    pout, _ = product_run(ren, sdf, col, var, *rays, device=device)
    oout = oracle["placement"]
    dz = (pout["z_vals"] - oout["z_vals"].detach()).abs().max(dim=1)[0]
    # fp32 round-off in the coarse SDF moves inverse-CDF samples by up to ~1e-3 even between the oracle's own
    # fp32 and fp64 runs (measured: DESIGN.md 'parity definition'); flips show up as much larger jumps.
    rep = {"case": oracle["name"], "R": R, "placement_frac_3e-3": (dz < 3e-3).float().mean().item(),
           "placement_median_dz": dz.median().item(), "placement_max_dz": dz.max().item()}
    dc = (pout["extra_color_fine"] - oout["extra_color_fine"].detach()).abs().max(dim=1)[0]
    rep["full_render_frac_rays_1e-3"] = (dc < 1e-3).float().mean().item()

    # (2) fine pass + backward on the oracle's depths
    oout2, ograds = oracle["fine"], oracle["grads"]
    pout2, pgrads = product_run(ren, sdf, col, var, *rays, cot=oracle["cot"], z_vals=oracle["z"], device=device)
    rep["out_err"] = {k: rel_to_max(pout2[k], oout2[k]) for k in COT_KEYS + ["mid_z_vals", "inside_sphere"]}
    rep["grad_err"] = {k: rel_to_max(pgrads[k], ograds[k]) for k in ograds}
    rep["worst_out"] = max(rep["out_err"].values())
    rep["worst_grad"] = max(rep["grad_err"].values())
    rep["grad_rel_l2"] = flat_rel_l2(pgrads, ograds)
    rep["engine"] = engine
    rep["oracle_dtype"] = oracle["oracle_dtype"]
    # bars (north_star: 1e-3 relative on the rendered outputs; gradients: VERDICT r1 asks <= 1e-3 rel-L2):
    #   fine pass on identical depths: every output within OUT_BAR (rel-to-max), flat gradient within 1e-3 rel-L2;
    #   full pipeline (own placement): >= 99 % of rays within 1e-3 in colour, >= 97 % within 3e-3 in depth -- the
    #   remainder are inverse-CDF bin flips, which the reference's own fp32 vs fp64 runs also show (DESIGN.md 5).
    out_bar = 1e-4 if engine == 0 else 1e-3
    rep["ok"] = (rep["worst_out"] < out_bar and rep["grad_rel_l2"] < 1e-3 and rep["placement_frac_3e-3"] >= 0.97
                 and rep["full_render_frac_rays_1e-3"] >= 0.99)
    log_parity("run_case", {k: rep[k] for k in ("case", "engine", "R", "oracle_dtype", "worst_out", "worst_grad",
                                                "grad_rel_l2", "placement_frac_3e-3", "placement_max_dz",
                                                "full_render_frac_rays_1e-3")})
    return rep
