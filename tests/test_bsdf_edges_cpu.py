"""CPU tests of the BSDF restatement (tests/bsdf_reference64.py) and of the oracle at the BSDFs' edges.

The restatement is checked against the reference fixtures before it is trusted; then the oracle -- the checker the GPU tests fall back
to -- is held to it on the adversarial tuples of every configuration, old and new."""
import numpy as np
import pytest

import bsdf_reference64 as R
from golden_inputs import BSDF_CONFIGS, GLASS, MICROFACET, MIRROR, PLASTIC, bsdf_inputs, material_desc
from oracle_binding import oracle_context
from parity import frac_within, golden, make_isects, rel_err

# what sample() of the microfacet family returns is ill-conditioned in the sampled direction (tests/test_large_batches.py): the
# same gate the kernel has in tests/test_gpu_parity.py -- at most one of the 512 fixture tuples beyond 1e-5, none beyond 5e-4
MICROFACET_SAMPLE_GATE = (1.5, 5e-4)


def _inside(v, env):
    v = np.asarray(v, np.float64)
    with np.errstate(invalid="ignore"):
        ok = ((v >= env["lo"]) & (v <= env["hi"])) | (np.isnan(v) & np.isnan(env["f32"]))
    return ok.all(-1) if ok.ndim > 1 else ok


@pytest.mark.parametrize("name", sorted(BSDF_CONFIGS))
def test_restatement_matches_reference_fixtures(name):
    cfg = BSDF_CONFIGS[name]
    g = golden("bsdf_" + name)
    wo, ng, ns, uv, wi, xi = bsdf_inputs(name, len(g["pdf"]))
    ef, ep = R.eval_envelope(cfg, wo, ng, ns, uv, wi)
    for key, env in (("f", ef), ("pdf", ep)):
        # float32 mode: every tuple within 1e-5, like the kernel
        ok, e = frac_within(env["f32"], g[key])
        assert ok == 1.0, (name, key, float(e.max()))
        # float64 mode: the reference inside the envelope everywhere, within 1e-5 of the float64 answer where the envelope is narrow.
        # (Not everywhere: D of a narrow lobe near the mirror direction moves by 1e-3 between float32 and float64 -- 1 - y^2 of a
        # float32 y near 1 -- and the reference is the float32 computation.)
        assert _inside(g[key], env).all(), (name, key, np.where(~_inside(g[key], env))[0][:5])
        well = R.envelope_ulps(env) < 10
        e64 = rel_err(env["f64"], g[key])
        e64 = e64.max(-1) if e64.ndim > 1 else e64
        assert (e64[well] <= 1e-5).all(), (name, key, float(e64[well].max()))
    sw, sp, _ = R.sample_envelope(cfg, wo, ng, ns, uv, xi)
    st, _ = R.eval_envelope(cfg, wo, ng, ns, uv, np.ascontiguousarray(g["sample_wi"])) if cfg["type"] not in (MIRROR, GLASS) else (None, None)
    if st is None:
        st = R.sample_envelope(cfg, wo, ng, ns, uv, xi)[2]
    for key, env in (("sample_wi", sw), ("sample_pdf", sp)):
        ok, e = frac_within(env["f32"], g[key])
        if cfg["type"] in (MICROFACET, PLASTIC):
            n_bad, cap = MICROFACET_SAMPLE_GATE
            assert ok >= 1.0 - n_bad / len(e) and e.max() <= cap, (name, key, ok, float(e.max()))
        else:
            assert ok == 1.0, (name, key, float(e.max()))
        assert _inside(g[key], env).all(), (name, key, np.where(~_inside(g[key], env))[0][:5])
    # the reference's throughput is f at its own sampled direction (delta BSDFs: the sample itself)
    assert _inside(g["sample_throughput"], st).all(), (name, np.where(~_inside(g["sample_throughput"], st))[0][:5])


# outputs the float32 mode computes with no libm call at all: these must be the oracle's bits
_NO_LIBM = {"lambertian": ("f", "pdf"), "lambertian_emissive": ("f", "pdf"), "lambertian_checker": ("f", "pdf"),
            "mirror": ("f", "pdf", "sample_wi", "sample_pdf", "sample_throughput"),
            "ggx_01": ("f", "pdf"), "ggx_05": ("f", "pdf"), "plastic_ggx": ("f", "pdf")}
_NO_LIBM.update({n: ("f", "pdf", "sample_wi", "sample_pdf", "sample_throughput") for n in BSDF_CONFIGS if n.startswith("glass")})


def _oracle(cfg, wo, ng, ns, uv, wi, xi):
    o = oracle_context()
    mat = o.add_material(material_desc(cfg, o))
    isects = make_isects(wo, ng, ns, uv, mat)
    f, pdf = o.bsdf_eval(mat, isects, wi)
    swi, spdf, sthr = o.bsdf_sample(mat, isects, xi)
    return dict(f=f, pdf=pdf, sample_wi=swi, sample_pdf=spdf, sample_throughput=sthr)


@pytest.mark.parametrize("name", sorted(_NO_LIBM))
def test_float32_restatement_is_the_oracle_bit_for_bit_without_libm(name):
    cfg = BSDF_CONFIGS[name]
    wo, ng, ns, uv, wi, xi = bsdf_inputs(name, 512)
    got = _oracle(cfg, wo, ng, ns, uv, wi, xi)
    f, pdf = R.bsdf_eval(cfg, wo, ng, ns, uv, wi, "float32")
    swi, spdf, sthr = R.bsdf_sample(cfg, wo, ng, ns, uv, xi, "float32")
    mine = dict(f=f, pdf=pdf, sample_wi=swi, sample_pdf=spdf, sample_throughput=sthr)
    for key in _NO_LIBM[name]:
        a, b = np.asarray(got[key], np.float32), np.asarray(mine[key], np.float32)
        same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
        assert same.all(), (name, key, np.where(~same.reshape(len(a), -1).all(-1))[0][:5])


def test_edge_inputs_cover_every_listed_case():
    tags = set()
    for cfg in R.ALL_CONFIGS.values():
        tags |= set(R.edge_inputs(cfg)[6])
    assert {"wo=ns", "wo=-ns", "wi=-wo", "mirror wi", "grazing wo", "grazing wi", "grazing both", "glass inside", "xi=R", "ns!=ng",
            "ns!=ng flipped", "snap", "snap wi", "snap ns", "s=0", "lambda a=1.6", "xi edge", "random"} <= tags
    xi = np.concatenate([R.edge_inputs(R.ALL_CONFIGS[n])[5] for n in ("plastic_dragon", "glass_15")])
    for v in (0.0, np.float32(1 - 2.0 ** -24), np.float32(0.5), np.float32(0.5 - 2.0 ** -24), np.float32(0.5 + 2.0 ** -24)):
        assert (xi == v).any(), v


@pytest.mark.parametrize("name", sorted(R.ALL_CONFIGS))
def test_oracle_within_the_restatement_on_adversarial_tuples(name):
    """the checker itself: NaN / inf pattern and sign as the float32 restatement, well-conditioned outputs within 1e-5 of float64,
    everything else inside the envelope"""
    cfg = R.ALL_CONFIGS[name]
    wo, ng, ns, uv, wi, xi, tags = R.edge_inputs(cfg)
    got = _oracle(cfg, wo, ng, ns, uv, wi, xi)
    fails = R.judge(cfg, (wo, ng, ns, uv, wi, xi), got)
    assert not fails, {k: [(tags[i], r) for i, r in v[:4]] for k, v in fails.items()}


def test_alpha_zero_is_pinned():
    """alpha = 0 passes ptc_add_material.  Pinned, not changed.  Beckmann: D = exp(-tan^2 * inf) / (pi * 0 * cos^4) = 0 / 0 is NaN for
    every half vector off the horizon, so f and pdf are NaN wherever the lobe is evaluated.  GGX: D = 0 / (pi cos^4 tan^4) is 0 except at
    wh = n, where it is 0 / 0; the sampler only returns wh = n, so every sampled pdf is NaN."""
    wo = np.array([[0.6, 0.8, 0.0], [0.0, 1.0, 0.0]], np.float32)
    ns = np.array([[0.0, 1.0, 0.0]] * 2, np.float32)
    uv = np.zeros((2, 2), np.float32)
    mirror = np.array([[-0.6, 0.8, 0.0], [0.0, 1.0, 0.0]], np.float32)
    other = np.array([[0.0, 0.8, 0.6], [0.6, 0.8, 0.0]], np.float32)
    xi = np.full((2, 3), 0.3, np.float32)
    for name in ("beckmann_0", "ggx_0"):
        cfg = R.ALL_CONFIGS[name]
        got = _oracle(cfg, wo, ns, ns, uv, mirror, xi)
        for mode in ("float32", "float64"):
            f, pdf = R.bsdf_eval(cfg, wo, ns, ns, uv, mirror, mode)
            assert np.isnan(f).all() and np.isnan(pdf).all(), (name, mode, f, pdf)
            f, pdf = R.bsdf_eval(cfg, wo, ns, ns, uv, other, mode)
            if name == "ggx_0":
                assert (f == 0).all() and (pdf == 0).all(), (mode, f, pdf)
            else:
                assert np.isnan(f).all() and np.isnan(pdf).all(), (mode, f, pdf)
            assert np.isnan(R.bsdf_sample(cfg, wo, ns, ns, uv, xi, mode)[1]).all()
        assert np.isnan(got["f"]).all() and np.isnan(got["pdf"]).all() and np.isnan(got["sample_pdf"]).all()


def test_axis_snap_makes_narrow_beckmann_pdfs_integrate_above_one():
    """The +-0.9999 axis snap of tfSinPhi replaces sin(phi) by 0 for half vectors within 0.81 degrees of the normal, so Beckmann's D
    there is exp(-tan^2 cos^2(phi) / alpha^2) instead of exp(-tan^2 / alpha^2).  A lobe narrower than the snap cone reports a pdf whose
    integral exceeds 1 by far, while the sampler draws the true Beckmann distribution; without the snap the same quadrature gives 1."""
    for name, lo, hi in (("beckmann_1e-4", 100.0, 300.0), ("beckmann_0005", 2.5, 4.0), ("beckmann_05", 0.97, 1.0 + 1e-3)):
        cfg = R.ALL_CONFIGS[name]
        snapped = R.upper_pdf_integral(cfg, 0.0)
        plain = R.upper_pdf_integral(cfg, 0.0, snap=2.0)
        assert lo <= snapped <= hi, (name, snapped)
        assert abs(plain - 1.0) < 2e-3 or name == "beckmann_05", (name, plain)


def test_restatement_pdf_integrals():
    """Lambertian and Oren-Nayar pdfs integrate to 1 over the upper hemisphere at every incidence (Oren-Nayar reports pdf 1 BELOW the
    surface, Q12, which is why only the upper hemisphere counts); the others to at most 1"""
    for name in ("lambertian", "oren_nayar_1"):
        for th in (0.0, 0.8, 1.5):
            assert abs(R.upper_pdf_integral(R.ALL_CONFIGS[name], th) - 1.0) < 1e-3, (name, th)
    for name in ("ggx_0005", "ggx_1", "beckmann_2", "plastic_ggx"):
        for th in (0.0, 0.8, 1.5):
            assert R.upper_pdf_integral(R.ALL_CONFIGS[name], th) <= 1.0 + 1e-3, (name, th)


def test_near_normal_wo_reaches_clampf_with_nan():
    """clampf = fminf(hi, fmaxf(v, lo)) sends NaN to lo (include/util.h:39-41).  On the adversarial tuples this is observable in one
    place only: wo within 1e-23 of the normal, where makeFrame's tangent axes are 0 / 0, every local vector is NaN, cartToSph's theta is
    acos(-1) = pi and Oren-Nayar's f stays finite.  A clampf that kept the NaN would make that f NaN; the oracle keeps it finite."""
    cfg = R.ALL_CONFIGS["oren_nayar_03"]
    wo, ng, ns, uv, wi, xi, tags = R.edge_inputs(cfg)
    k = tags == "near-normal wo"
    args = (wo[k], ng[k], ns[k], uv[k], wi[k])
    f, pdf = R.bsdf_eval(cfg, *args, "float32")
    assert np.isfinite(f).all() and np.isnan(pdf).all()
    assert np.isfinite(_oracle(cfg, *args, xi[k])["f"]).all()
    keep = R.clampf
    try:
        R.clampf = lambda v, lo, hi: np.where(np.isnan(v), v, keep(v, lo, hi))
        assert np.isnan(R.bsdf_eval(cfg, *args, "float32")[0]).all()
    finally:
        R.clampf = keep
