"""GPU parity tests of the NeuS path: CUDA (through the C ABI / product modules) vs the CPU oracle."""
import os

import pytest
import torch

import util_neus as U

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,bg,anneal", [("tiny", "ray", 1.0), ("tiny", "white", 0.3), ("skiplast", "none", 0.0),
                                             ("shipped", "ray", 1.0), ("b2", "white", 1.0)])
def test_synthetic_case_matches_oracle(name, bg, anneal):
    rep = U.run_case_gpu_vs_oracle(name, bg_kind=bg, anneal=anneal)
    print(rep)
    assert rep["worst_out"] < 1e-4, rep          # fp32 engine: an order below the north_star bar (measured ~4e-6)
    assert rep["grad_rel_l2"] < 1e-3, rep
    assert rep["worst_grad"] < 2e-3, rep
    assert rep["placement_frac_3e-3"] >= 0.97, rep
    assert rep["full_render_frac_rays_1e-3"] >= 0.99, rep


def test_chunked_equals_single_chunk():
    """Multi-chunk rendering (recompute-in-backward path) must equal the single-chunk path."""
    a = U.run_case_gpu_vs_oracle("tiny", chunk=4096, R=50)
    b = U.run_case_gpu_vs_oracle("tiny", chunk=16, R=50)
    assert b["ok"], b
    assert abs(a["worst_out"] - b["worst_out"]) < 1e-4
    assert b["grad_rel_l2"] < 1e-3


def test_chunked_tcgen05_engine_at_scale():
    """Multi-chunk recompute path on engine 1 at a realistic size: 8192 rays of the shipped-size nets in chunks of 2048
    against ONE chunk of 8192 (same kernels, different chunking; the oracle cannot hold 8 k rays in seconds)."""
    sdf_kw, col_kw, ren_kw, _ = U.CASES["shipped"]
    sp, cp = U.synth_state(sdf_kw, col_kw, 2)
    R = 8192
    o, d, near, far, jit = U.make_rays(R, 11)
    g = torch.Generator().manual_seed(12)
    bg = torch.rand(R, 1, generator=g)
    res = []
    for chunk in (8192, 2048):
        sdf, col, var, ren = U.build_product(sdf_kw, col_kw, ren_kw, sp, cp, 0.3, "cuda", engine=1, chunk=chunk)
        out, _ = U.product_run(ren, sdf, col, var, o, d, near, far, jit, bg, 1.0)
        cot = U.cotangents(out, seed=13)
        out2, grads = U.product_run(ren, sdf, col, var, o, d, near, far, jit, bg, 1.0, cot=cot, z_vals=out["z_vals"])
        res.append((out, out2, grads))
    (oa, oa2, ga), (ob, ob2, gb) = res
    assert torch.equal(oa["z_vals"], ob["z_vals"])          # placement is per ray: chunking must not change it
    for k in ("color_fine", "extra_color_fine", "weights", "gradients", "cdf_fine"):
        assert U.rel_to_max(ob2[k], oa2[k]) < 1e-5, k
    # gradient_error normalises over ALL rays of the call
    assert U.rel_to_max(ob2["gradient_error"], oa2["gradient_error"]) < 1e-5
    l2 = U.flat_rel_l2(gb, ga)
    U.log_parity("chunked_engine1_8192", {"grad_rel_l2_chunked_vs_single": l2})
    assert l2 < 1e-4, l2          # summation order of the per-chunk weight gradients differs


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("name", ["cfg1", "small", "shipped"])
def test_golden_reference_vectors(name, engine):
    """Outputs and parameter gradients recorded from the UNMODIFIED reference (tests/golden), both engines.
    ``shipped`` = pretrained_models/zero_beta_stand_pose.pth (4x256 + 2x256, variance 0.6277 -> inv_s ~ 532): the
    weights the reference actually trains from, and the regime where reduced precision breaks RGB parity
    (SURVEY Appendix C) -- the tcgen05 engine (two-term bf16 split) has to hold the 1e-3 bar THERE."""
    b = torch.load(os.path.join(U.GOLDEN, f"neus_{name}.pt"), map_location="cpu", weights_only=False)
    sdf, col, var, ren = U.build_product(b["sdf_kw"], b["col_kw"], b["ren_kw"], b["sdf_state"], b["col_state"],
                                         b["variance"], "cuda", engine=engine)
    cot = b["loss_weights"]
    out, grads = U.product_run(ren, sdf, col, var, b["rays_o"], b["rays_d"], b["near"], b["far"], b["jitter"],
                               b["background"], b["cos_anneal"], cot=cot, z_vals=b["z_vals"])
    errs = {k: U.rel_to_max(out[k], ref) for k, ref in b["out"].items()}
    gerrs = {k: U.rel_to_max(grads[k], ref) for k, ref in b["grads"].items()}
    l2 = U.flat_rel_l2(grads, b["grads"])
    # placement from scratch against the reference's own depths, and the colours that come out of it
    out2, _ = U.product_run(ren, sdf, col, var, b["rays_o"], b["rays_d"], b["near"], b["far"], b["jitter"],
                            b["background"], b["cos_anneal"])
    dz = (out2["z_vals"] - b["z_vals"]).abs().max(dim=1)[0]
    dc = torch.maximum((out2["extra_color_fine"] - b["out"]["extra_color_fine"]).abs().max(dim=1)[0],
                       (out2["color_fine"] - b["out"]["color_fine"]).abs().max(dim=1)[0])
    rec = {"golden": name, "engine": engine, "worst_out": max(errs.values()), "worst_out_key": max(errs, key=errs.get),
           "rgb_err": max(errs["color_fine"], errs["extra_color_fine"]), "worst_grad": max(gerrs.values()),
           "grad_rel_l2": l2, "placement_frac_3e-3": (dz < 3e-3).float().mean().item(),
           "placement_max_dz": dz.max().item(), "full_render_frac_rays_1e-3": (dc < 1e-3).float().mean().item(),
           "full_render_max_abs": dc.max().item()}
    print(rec)
    U.log_parity("golden_reference_vectors", rec)
    out_bar = 1e-4 if engine == 0 else 1e-3
    for k, e in errs.items():
        assert e < out_bar, (k, e)
    assert l2 < 1e-3, l2
    assert rec["placement_frac_3e-3"] >= 0.97, rec
    assert rec["full_render_frac_rays_1e-3"] >= 0.99, rec


def test_sdf_query_matches_oracle():
    sdf_kw, col_kw, ren_kw, _ = U.CASES["shipped"]
    sconf, cconf, rconf = U.confs_from_kw(sdf_kw, col_kw, ren_kw)
    sp, cp = U.synth_state(sdf_kw, col_kw, 3)
    sdf, col, var, ren = U.build_product(sdf_kw, col_kw, ren_kw, sp, cp, 0.3, "cuda")
    pts = (torch.rand(5000, 3) - 0.5) * 2
    got = sdf.sdf(pts.cuda()).cpu()
    from oracle import neus
    want = neus.sdf_value(sp, sconf, pts)
    assert U.rel_to_max(got, want) < 1e-5


# five full waves of 128-point tiles on 148 SMs plus a ragged tile: the busiest chain CTA walks 6 tiles
P_PERSISTENT = 5 * 148 * 128 + 77


def _chain_net(name, seed):
    """(sdf_kw, col_kw, ren_kw, sdf_state, col_state, variance): a synthetic case or the weights of a golden vector."""
    if name in U.CASES:
        sdf_kw, col_kw, ren_kw, _ = U.CASES[name]
        sp, cp = U.synth_state(sdf_kw, col_kw, seed)
        return sdf_kw, col_kw, ren_kw, sp, cp, 0.3
    b = torch.load(os.path.join(U.GOLDEN, f"neus_{name}.pt"), map_location="cpu", weights_only=False)
    return b["sdf_kw"], b["col_kw"], b["ren_kw"], b["sdf_state"], b["col_state"], b["variance"]


def _chain_query_errors(name, P, chunk=4096):
    """sdf_query of engine 1 on P points against the fp64 oracle, with the fused chain (default) and with the
    layer-by-layer launches (AVC_FUSED_CHAIN=0).  Returns {variant: rel-to-max error}."""
    sdf_kw, col_kw, ren_kw, sp, cp, variance = _chain_net(name, 5)
    sconf, cconf, rconf = U.confs_from_kw(sdf_kw, col_kw, ren_kw)
    sdf, col, var, ren = U.build_product(sdf_kw, col_kw, ren_kw, sp, cp, variance, "cuda", engine=1, chunk=chunk)
    pts = (torch.rand(P, 3, generator=torch.Generator().manual_seed(P)) - 0.5) * 2
    from oracle import neus
    want = neus.sdf_value({k: v.double() for k, v in sp.items()}, sconf, pts.double())
    errs = {}
    saved = os.environ.get("AVC_FUSED_CHAIN")
    try:
        for variant, env in (("fused", None), ("layered", "0")):
            if env is None:
                os.environ.pop("AVC_FUSED_CHAIN", None)
            else:
                os.environ["AVC_FUSED_CHAIN"] = env
            errs[variant] = U.rel_to_max(sdf.sdf(pts.cuda()).cpu(), want)
    finally:
        if saved is None:
            os.environ.pop("AVC_FUSED_CHAIN", None)
        else:
            os.environ["AVC_FUSED_CHAIN"] = saved
    return errs


@pytest.mark.parametrize("name,P", [("tiny", 77), ("tiny", 5000), ("skiplast", 1000), ("shipped", 4099), ("b2", 20000),
                                    ("tiny", P_PERSISTENT), ("skiplast", P_PERSISTENT), ("shipped", P_PERSISTENT),
                                    ("b2", P_PERSISTENT), ("cfg1", P_PERSISTENT)])
def test_fused_chain_sdf_query_matches_oracle(name, P):
    """engine 1 without a stash (sample placement, SDFNetwork.sdf) runs the whole value chain of a 128-point tile in ONE
    kernel (csrc/avc_chain.cu: activations resident in shared memory, sdf head folded into the last epilogue).  Covered:
    widths 48 / 64 / 256, the skip concat inside the chain and at the head, ragged last tile, P < one tile, and at
    P_PERSISTENT several tiles per CTA (the A tile is reloaded and the weight ring runs on across tiles) for chains of
    4 and 9 layers, among them nets whose last chain layer has K <= 64 (tiny, skiplast, cfg1).  The layer-by-layer
    tcgen05 launches (AVC_FUSED_CHAIN=0) are held to the same bar."""
    errs = _chain_query_errors(name, P)
    U.log_parity("fused_chain_sdf_query", {"case": name, "P": P, "tiles_per_cta": U.chain_tiles_per_cta(P),
                                           "rel_to_max": errs["fused"], "rel_to_max_layered": errs["layered"]})
    if P == P_PERSISTENT:
        assert U.chain_tiles_per_cta(P) >= 5, U.chain_tiles_per_cta(P)
    for variant, err in errs.items():
        assert err < 5e-5, (variant, err)      # two-term bf16 split operands (~16 mantissa bits); measured ~1e-5


def test_sdf_query_many_chunks():
    """sdf_query splits P into chunks of max_rays_per_chunk * S points (avc_neus_sdf_query's p0 loop): 16 rays x 64
    samples = 1024 points a chunk, 93 chunks with a ragged last one, each encoded and run through the chain."""
    P = P_PERSISTENT
    errs = _chain_query_errors("shipped", P, chunk=16)
    U.log_parity("fused_chain_sdf_query", {"case": "shipped", "P": P, "chunk_points": 16 * 64,
                                           "rel_to_max": errs["fused"], "rel_to_max_layered": errs["layered"]})
    assert -(-P // (16 * 64)) >= 90
    for variant, err in errs.items():
        assert err < 5e-5, (variant, err)


@pytest.mark.parametrize("name,bg,anneal", [("tiny", "ray", 1.0), ("skiplast", "none", 0.3), ("shipped", "ray", 1.0),
                                             ("b2", "white", 1.0)])
def test_tcgen05_engine_matches_oracle(name, bg, anneal):
    """engine 1: tcgen05 tiles with two-term bf16 split operands (3 MMAs per product).  The bar is the
    north_star's: rendered outputs within 1e-3 relative; flat gradient within 1e-3 rel-L2."""
    rep = U.run_case_gpu_vs_oracle(name, bg_kind=bg, anneal=anneal, engine=1)
    print({k: rep[k] for k in ("case", "worst_out", "worst_grad", "placement_frac_3e-3", "placement_max_dz",
                               "full_render_frac_rays_1e-3")})
    assert rep["worst_out"] < 1e-3, rep
    assert rep["grad_rel_l2"] < 1e-3, rep          # measured 2e-5 .. 4e-5 (profiles/r2_parity.json)
    # per-tensor rel-to-max is dominated by tensors whose whole gradient is ~1e-4 of the largest one (measured up to
    # 1.1e-2 on such a tensor at b2 while the flat gradient is within 2e-5): reported, loosely bounded
    assert rep["worst_grad"] < 5e-2, rep
    assert rep["placement_frac_3e-3"] >= 0.97, rep
    assert rep["full_render_frac_rays_1e-3"] >= 0.99, rep
