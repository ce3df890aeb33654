"""The render at the benchmark's size, where every persistent kernel walks several tiles per CTA.

At 512 rays x 128 samples = 65 536 fine points the tcgen05 NT launches run 7 row tiles per CTA (the TMEM accumulator
ring of 4 wraps), the weight-gradient TN CTAs reduce 14 k-blocks through their 2-4 stages and the fused value chain of
the sample placement reloads its A tile for every further tile.  The small synthetic cases and golden vectors run one
tile per CTA and cannot see a defect that only appears from a CTA's second or fifth tile on; these cases can:

* the benchmark-scale fine pass and backward against the fp64 oracle (both engines, and the single-pass precision
  options of engine 1);
* rays in reversed order: at 128 samples one ray is one fine tile, so reversing moves every tile between the first and
  the last position of its CTA; per-ray results must not change;
* narrow nets (BN = 64 tiles, chains whose last layer has one k-block) at 4096 rays.

The oracle is computed once per module (fixture), never at import."""
import pytest
import torch

import util_neus as U

pytestmark = pytest.mark.gpu

R_BENCH = 512          # rays of the benchmark (bench.py): b2 samples 64 + 64 per ray


@pytest.fixture(scope="module")
def b2_oracle():
    return U.oracle_case("b2", seed=0, bg_kind="ray", anneal=1.0, R=R_BENCH, oracle_dtype=torch.float64)


def _fine_points(name, R):
    ren_kw = U.CASES[name][2]
    return R * (ren_kw["n_samples"] + ren_kw["n_importance"])


def _log(test, rep, **extra):
    rec = {k: rep[k] for k in ("case", "engine", "R", "oracle_dtype", "worst_out", "worst_grad", "grad_rel_l2",
                               "placement_frac_3e-3", "placement_max_dz", "full_render_frac_rays_1e-3")}
    rec["rgb_err"] = max(rep["out_err"]["color_fine"], rep["out_err"]["extra_color_fine"])
    U.log_parity(test, dict(rec, **extra))


@pytest.mark.parametrize("engine", [0, 1])
def test_benchmark_scale_matches_oracle(b2_oracle, engine):
    """b2 (8 x 256 SDF + 4 x 256 colour, 64 + 64 samples) at 512 rays: fine pass and backward on the oracle's depths
    against fp64, and the full pipeline's placement against the oracle's fp32 placement."""
    tiles = U.nt_tiles_per_cta(_fine_points("b2", R_BENCH), 256)
    assert tiles > 4, tiles                          # the 4 TMEM accumulators of the NT kernel are reused
    rep = U.run_case_gpu_vs_oracle("b2", engine=engine, oracle=b2_oracle)
    _log("persistent_benchmark_scale", rep, nt_tiles_per_cta=tiles)
    assert rep["worst_out"] < (1e-4 if engine == 0 else 1e-3), rep
    assert rep["grad_rel_l2"] < 1e-3, rep
    assert rep["placement_frac_3e-3"] >= 0.97, rep
    assert rep["full_render_frac_rays_1e-3"] >= 0.99, rep


def test_single_pass_precision_options(b2_oracle):
    """color_products = 1, wgrad_products = 1: the NPROD = 1 NT and TN launches with their real epilogues.  DESIGN
    3.1 documents 1e-3 .. 2.5e-3 rel-L2 for the gradient of these options; the bars here catch a broken kernel, they do
    not judge that precision loss."""
    rep = U.run_case_gpu_vs_oracle("b2", engine=1, oracle=b2_oracle, color_products=1, wgrad_products=1)
    _log("persistent_single_pass_options", rep)
    assert rep["worst_out"] < 1e-3, rep
    assert rep["grad_rel_l2"] < 5e-3, rep


def test_ray_permutation_invariance():
    """engine 1, b2 at 512 rays, rendered in order and reversed (jitter, background and the fixed depths permuted
    alike).  No kernel on the path depends on a row's position, so every per-ray output, and the placed depths, must be
    bitwise equal; the gradient_error scalar and the parameter gradient are sums over all rays whose fp32 order
    changes with the permutation."""
    sdf_kw, col_kw, ren_kw, _ = U.CASES["b2"]
    sp, cp = U.synth_state(sdf_kw, col_kw, 0)
    R = R_BENCH
    assert U.nt_tiles_per_cta(_fine_points("b2", R), 256) > 4
    o, d, near, far, jit = U.make_rays(R, 21)
    bg = torch.rand(R, 1, generator=torch.Generator().manual_seed(22))
    perm = torch.arange(R - 1, -1, -1)
    sdf, col, var, ren = U.build_product(sdf_kw, col_kw, ren_kw, sp, cp, 0.3, "cuda", engine=1)
    rays = (o, d, near, far, jit, bg)
    rays_p = tuple(t[perm] for t in rays)

    a, _ = U.product_run(ren, sdf, col, var, *rays, 1.0)
    b, _ = U.product_run(ren, sdf, col, var, *rays_p, 1.0)
    cot = U.cotangents(a, seed=23)
    cot_p = {k: (v[perm] if v.dim() > 0 and v.shape[0] == R else v) for k, v in cot.items()}
    a2, ga = U.product_run(ren, sdf, col, var, *rays, 1.0, cot=cot, z_vals=a["z_vals"])
    b2, gb = U.product_run(ren, sdf, col, var, *rays_p, 1.0, cot=cot_p, z_vals=a["z_vals"][perm])

    diffs, scalars = {}, {}
    for tag, x, y in (("placement", a, b), ("fixed_depths", a2, b2)):
        for k, v in x.items():
            if v is None:
                continue
            if v.dim() > 0 and v.shape[0] == R:
                diffs[f"{tag}.{k}"] = (v[perm].double() - y[k].double()).abs().max().item()
            else:
                scalars[f"{tag}.{k}"] = U.rel_to_max(y[k], v)
    l2 = U.flat_rel_l2(gb, ga)
    U.log_parity("persistent_ray_permutation", {"max_abs_per_ray": max(diffs.values()),
                                                "worst_key": max(diffs, key=diffs.get), "scalars_rel": scalars,
                                                "grad_rel_l2": l2})
    nonzero = {k: v for k, v in diffs.items() if v != 0.0}
    assert not nonzero, nonzero
    for k, e in scalars.items():
        assert e < 1e-5, (k, e)
    assert l2 < 1e-5, l2


@pytest.mark.parametrize("name,bg,anneal", [("tiny", "ray", 1.0), ("skiplast", "none", 0.3)])
def test_narrow_net_many_tiles(name, bg, anneal):
    """48- and 64-wide nets at 4096 rays: the placement runs the fused chain (last chain layer K <= 64) over 64 k /
    98 k coarse points, and the fine pass the BN = 64 NT tiles at 7 tiles per CTA."""
    R = 4096
    chain = U.chain_tiles_per_cta(R * U.CASES[name][2]["n_samples"])
    nt = U.nt_tiles_per_cta(_fine_points(name, R), U.CASES[name][0]["d_hidden"])
    assert chain >= 2 and nt > 4, (chain, nt)
    rep = U.run_case_gpu_vs_oracle(name, engine=1, bg_kind=bg, anneal=anneal, R=R, oracle_dtype=torch.float64)
    _log("persistent_narrow_net", rep, chain_tiles_per_cta=chain, nt_tiles_per_cta=nt)
    assert rep["worst_out"] < 1e-3, rep
    assert rep["grad_rel_l2"] < 1e-3, rep
    assert rep["worst_grad"] < 5e-2, rep
    assert rep["placement_frac_3e-3"] >= 0.97, rep
    assert rep["full_render_frac_rays_1e-3"] >= 0.99, rep
