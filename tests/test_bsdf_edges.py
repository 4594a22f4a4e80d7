"""GPU tests of bsdfEval / bsdfSample (pathed_b200/csrc/shading.cuh, through the C ABI) at their edges: adversarial tuples against the
restatement (tests/bsdf_reference64.py) and the oracle, sampling against the pdf (chi^2), delta BSDFs, finiteness."""
import numpy as np
import pytest
from scipy import stats

import bsdf_reference64 as R
from golden_inputs import BECKMANN, MICROFACET, MIRROR, PLASTIC, material_desc, uniform_floats, unit_vectors
from oracle_binding import oracle_context
from parity import make_isects

pytestmark = pytest.mark.gpu


def _kernel(cfg):
    from pathed_b200 import create_context
    ctx = create_context(0)
    mat = ctx.add_material(material_desc(cfg, ctx))
    ctx.add_triangle_mesh([[0, 0, 0], [1, 0, 0], [0, 1, 0]], None, None, [[0, 1, 2]], mat)
    ctx.set_camera((0, 0, 5), (0, 0, 0), (0, 1, 0), 0.5, 8, 8)
    ctx.commit()
    return ctx, mat


def _run(api, mat, wo, ng, ns, uv, wi, xi):
    isects = make_isects(wo, ng, ns, uv, mat)
    f, pdf = api.bsdf_eval(mat, isects, wi)
    swi, spdf, sthr = api.bsdf_sample(mat, isects, xi)
    return dict(f=f, pdf=pdf, sample_wi=swi, sample_pdf=spdf, sample_throughput=sthr)


@pytest.mark.parametrize("name", sorted(R.ALL_CONFIGS))
def test_kernel_on_adversarial_tuples(name):
    """(a) finite / NaN / inf pattern and sign of every output as the float32 restatement's and the oracle's, (b) well-conditioned
    outputs (envelope below 10 ulp) within 1e-5 of float64, (c) every other finite output inside the envelope; the sampled throughput
    is judged as f at the kernel's own sampled direction"""
    cfg = R.ALL_CONFIGS[name]
    wo, ng, ns, uv, wi, xi, tags = R.edge_inputs(cfg)
    ctx, mat = _kernel(cfg)
    got = _run(ctx, mat, wo, ng, ns, uv, wi, xi)
    fails = R.judge(cfg, (wo, ng, ns, uv, wi, xi), got)
    assert not fails, {k: [(tags[i], r) for i, r in v[:4]] for k, v in fails.items()}
    o = oracle_context()
    want = _run(o, o.add_material(material_desc(cfg, o)), wo, ng, ns, uv, wi, xi)
    for key in ("f", "pdf", "sample_pdf", "sample_throughput", "sample_wi"):
        a, b = R._sign_class(got[key]), R._sign_class(want[key])
        diff = (a != b).reshape(len(wo), -1).any(-1)
        assert not diff.any(), (key, [(tags[i], got[key][i], want[key][i]) for i in np.where(diff)[0][:4]])


# ------------------------------------------------------------------------------------------------ sampling against the pdf
N_SAMPLES = 1 << 22
INCIDENCES = [(0.0, 0.0), (45.0, 0.0), (80.0, 0.0), (89.9, 0.0), (45.0, 0.3)]  # (theta_o in degrees, tilt of ng away from ns)
# (config, incidences).  Left out, by reason -- in each case the float32 restatement, used as the sampler, fails the same way, so the
# test could not tell a kernel error there:
# - alpha <= ~3e-4 (beckmann_1e-4, plastic_1e-4): the float32 sampler's sinT = sqrt(1 - cosT^2) is 0 for tan^2 < 2^-24, so every
#   sample is the exact mirror direction (test_narrow_lobes_sample_the_mirror_direction); at alpha = 0.005 and 0.02 (beckmann_0005,
#   beckmann_002) 1 + tan^2 and cosT^2 are rounded on a float32 grid that coarse against the lobe that 2^22 samples see the
#   quantisation (chi^2 442 on 191 dof for alpha = 0.02, the same value for kernel and restatement)
# - the glossy lobes at 89.9 degrees, beckmann_2 at 80 and beckmann_1 / ggx_1 off normal incidence: samples land right at the horizon
#   in cells to which the quadrature gives no mass
GLOSSY = ("beckmann_005", "beckmann_01", "beckmann_05", "ggx_0005", "ggx_002", "ggx_01", "plastic_ggx", "plastic_dragon")
CHI2_CASES = [(n, INCIDENCES) for n in ("lambertian", "oren_nayar_1")] + \
             [(n, [i for i in INCIDENCES if i[0] < 89]) for n in GLOSSY] + \
             [("beckmann_2", [i for i in INCIDENCES if i[0] < 60])] + [(n, INCIDENCES[:1]) for n in ("beckmann_1", "ggx_1")]
CHI2_CONFIGS = [n for n, _ in CHI2_CASES]
# the axis snap (test_bsdf_edges_cpu.py::test_axis_snap_makes_narrow_beckmann_pdfs_integrate_above_one): for a Beckmann lobe that
# reaches into the 0.81-degree snap cone eval's pdf is not the density the sampler draws from.  Their expected counts come from the
# unsnapped D; the pdf integral asserts the quirk by name
SNAP_QUIRK = {"beckmann_0005", "beckmann_002", "beckmann_005", "beckmann_1e-4", "plastic_1e-4"}
P_FAMILY = 1e-4
QUAD_REL = 1e-2


def _stratified_xi(n, seed):
    k = int(np.sqrt(n))
    i, j = np.meshgrid(np.arange(k), np.arange(k), indexing="ij")
    u = uniform_floats(seed, (n, 3)).astype(np.float64)
    xi = np.stack([(i.reshape(-1) + u[:, 0]) / k, (j.reshape(-1) + u[:, 1]) / k, u[:, 2]], 1)
    return np.ascontiguousarray(np.minimum(xi, 1 - 2.0 ** -24).astype(np.float32))


def _cell_masses(cfg, wo, ng, ns, F, s0, s1, p0, p1, snap, sub):
    """per (s, phi) cell: (mass of the restatement's eval pdf above the surface, mass the sampler puts below it, cut) -- cut: the cell
    straddles a discontinuity of the integrand (the horizon, or for Beckmann the edge of the axis snap)"""
    wi_l, dwi, wh, dwh = R.halfvector_cell_nodes(s0, s1, p0, p1, F @ wo[0].astype(np.float64), R.lobe_width(cfg), 4, sub)
    m, k = dwi.shape
    wi = np.asarray(wi_l.reshape(-1, 3) @ F, np.float32)
    rep = lambda a: np.repeat(a, m * k, 0)
    pdf = R.bsdf_eval(cfg, rep(wo), rep(ng), rep(ns), np.zeros((m * k, 2), np.float32), wi, "float64", snap=snap)[1].reshape(m, k)
    above = ((wi.astype(np.float64) @ ns[0].astype(np.float64)) >= 0).reshape(m, k)
    upper = (np.where(above, pdf, 0) * dwi).sum(1)
    below = np.zeros(m)
    if cfg["type"] in (MICROFACET, PLASTIC):
        # the sampler's mass below the surface, where eval reports pdf 0: the grid's own half vectors whose reflection of wo points
        # down, weighted by D(wh) |wh.y|; Plastic picks the microfacet lobe half the time
        with np.errstate(all="ignore"):
            d = R.mf_pdf(R._M(np.float64), cfg, (wh[..., 0], wh[..., 1], wh[..., 2]), snap)
        below = (np.where(~above, d, 0) * dwh).sum(1) * (0.5 if cfg["type"] == PLASTIC else 1.0)
    snapped = (np.abs(wh) >= R.SNAP).any(-1) if cfg.get("distribution") == BECKMANN and snap == R.SNAP else np.zeros_like(above)
    cut = (above.any(1) & ~above.all(1)) | (snapped.any(1) & ~snapped.all(1))
    return upper, below, cut


def _chi2_case(ctx, mat, cfg, theta_deg, tilt, xi):
    wo, ng, ns, F, se, pe, _, _ = R.halfvector_grid(cfg, np.radians(theta_deg), tilt)
    n_s, n_phi = len(se) - 1, len(pe) - 1
    # expected: float64 quadrature of the restatement's pdf over every (s, phi) cell; cells that straddle a discontinuity are
    # integrated again on an 8 x 8 finer grid
    snap = 2.0 if cfg.get("_name") in SNAP_QUIRK else R.SNAP
    S0, P0 = np.meshgrid(se[:-1], pe[:-1], indexing="ij")
    S1, P1 = np.meshgrid(se[1:], pe[1:], indexing="ij")
    S0, S1, P0, P1 = (a.reshape(-1) for a in (S0, S1, P0, P1))
    upper, below_cells, cut = _cell_masses(cfg, wo, ng, ns, F, S0, S1, P0, P1, snap, 1)
    if cut.any():
        upper[cut], below_cells[cut], _ = _cell_masses(cfg, wo, ng, ns, F, S0[cut], S1[cut], P0[cut], P1[cut], snap, 8)
    mass = upper.reshape(n_s, n_phi)
    below_mass = float(below_cells.sum())
    total = mass.sum() + below_mass
    assert abs(total - 1) < 2e-3, ("sampling density does not integrate to 1", total)
    # samples
    n = len(xi)
    wi, spdf, thr = ctx.bsdf_sample(mat, make_isects(np.repeat(wo, n, 0), np.repeat(ng, n, 0), np.repeat(ns, n, 0), np.zeros((n, 2), np.float32), mat), xi)
    wl = wi.astype(np.float64) @ F.T
    below = wl[:, 1] < 0
    s, phi = R.halfvector_coords(F @ wo[0].astype(np.float64), wl, R.lobe_width(cfg))
    si = np.clip(np.searchsorted(se, s) - 1, 0, n_s - 1)
    pi = np.clip(np.searchsorted(pe, phi) - 1, 0, n_phi - 1)
    # coarse bins: s panels merged into ~24 groups of equal expected mass, phi in 16 groups; the last bin is "below the surface"
    cum = np.cumsum(mass.sum(1)) / max(mass.sum(), 1e-300)
    s_group = np.minimum((cum * 24).astype(int), 23)
    p_group = np.arange(n_phi) * 16 // n_phi
    cell = (s_group[:, None] * 16 + p_group[None, :]).reshape(-1)
    nb = 24 * 16 + 1
    expected = np.append(np.bincount(cell, mass.reshape(-1), minlength=nb - 1), below_mass) * n / total
    observed = np.append(np.bincount(cell[si[~below] * n_phi + pi[~below]], minlength=nb - 1), below.sum()).astype(np.float64)
    approx = np.append(np.bincount(cell, cut, minlength=nb - 1) > 0, below_mass > 0)  # bins whose mass comes from refined cells
    small = expected < 20
    e = np.append(expected[~small], expected[small].sum())
    o = np.append(observed[~small], observed[small].sum())
    a = np.append(approx[~small], approx[small].any())
    assert e[-1] > 0 or o[-1] == 0, "samples where the pdf says none can be"
    # Pearson; bins whose cells straddle a discontinuity carry a variance floor for the quadrature's remaining error there
    var = e + np.where(a, (QUAD_REL * e) ** 2, 0)
    keep = e > 0
    chi2 = float(((o[keep] - e[keep]) ** 2 / var[keep]).sum())
    return chi2, int(keep.sum()) - 1, float(stats.chi2.sf(chi2, int(keep.sum()) - 1)), float(expected[:-1].sum() / n)


def test_sampling_matches_the_pdf():
    """chi^2 of 2^22 stratified samples per case, binned in half-vector coordinates scaled by the lobe width (ln(tan(theta_h) / w),
    phi_h), against float64 quadrature of the restatement's pdf; one bin for the mass the sampler puts below the surface.  Family-wise
    level 1e-4 (Sidak over all cases)."""
    cases = [(n, t, g) for n, inc in CHI2_CASES for t, g in inc]
    p_case = 1 - (1 - P_FAMILY) ** (1 / len(cases))
    xi = _stratified_xi(N_SAMPLES, 4321)
    worst = []
    for name, incidences in CHI2_CASES:
        cfg = dict(R.ALL_CONFIGS[name], _name=name)
        ctx, mat = _kernel(R.ALL_CONFIGS[name])
        for theta, tilt in incidences:
            chi2, dof, p, upper = _chi2_case(ctx, mat, cfg, theta, tilt, xi)
            print("%-14s theta %5.1f tilt %.1f: chi2 %9.1f dof %3d p %.3g (upper-hemisphere mass %.5f)" % (name, theta, tilt, chi2, dof, p, upper))
            worst.append((p, name, theta, tilt))
    assert min(worst)[0] >= p_case, (sorted(worst)[:5], p_case)


def test_kernel_pdf_integrates_to_one():
    """the kernel's own eval pdf, integrated on the half-vector quadrature grid over the upper hemisphere: 1 for Lambertian and
    Oren-Nayar, at most 1 for the others -- except the lobes narrower than the axis snap cone, which integrate far above 1 (named)"""
    for name in CHI2_CONFIGS + ["beckmann_1e-4", "plastic_1e-4", "beckmann_0005", "beckmann_002"]:
        cfg = R.ALL_CONFIGS[name]
        ctx, mat = _kernel(cfg)

        def evaluate(wo, ng, ns, uv, wi):
            return ctx.bsdf_eval(mat, make_isects(wo, ng, ns, uv, mat), wi)[1].astype(np.float64)
        for theta, tilt in INCIDENCES:
            got = R.upper_pdf_integral(cfg, np.radians(theta), tilt_ng=tilt, evaluate=evaluate)
            want = R.upper_pdf_integral(cfg, np.radians(theta), tilt_ng=tilt)
            if name in ("beckmann_1e-4", "plastic_1e-4", "beckmann_0005"):
                assert got > 1.5, (name, theta, got)  # axis snap quirk (its integrand is too ill-conditioned to compare closer)
                continue
            assert abs(got - want) <= 2e-3, (name, theta, got, want)  # float32 D of a narrow lobe vs float64
            if name in ("lambertian", "oren_nayar_1"):
                assert abs(got - 1) < 1e-3, (name, theta, got)
            elif name not in SNAP_QUIRK:  # beckmann_002 / 005 reach into the snap cone and may exceed 1 a little
                assert got <= 1 + 2e-3, (name, theta, got)


# ------------------------------------------------------------------------------------------------ delta BSDFs
def _fresnel64(cos_i, eta_i, eta_t):
    sin_t = eta_i / eta_t * np.sqrt(np.maximum(0, 1 - cos_i ** 2))
    cos_t = np.sqrt(np.maximum(0, 1 - sin_t ** 2))
    r_par = (eta_t * cos_i - eta_i * cos_t) / (eta_t * cos_i + eta_i * cos_t)
    r_perp = (eta_i * cos_i - eta_t * cos_t) / (eta_i * cos_i + eta_t * cos_t)
    return np.where(sin_t > 1, 1.0, 0.5 * (r_par ** 2 + r_perp ** 2))


@pytest.mark.parametrize("name", ["mirror", "glass_11", "glass_15", "glass_20", "glass_10", "glass_10001", "glass_24"])
def test_delta_directions_are_exact(name):
    """sampled directions are the exact (float64) reflection / refraction of wo within the sample envelope"""
    cfg = R.ALL_CONFIGS[name]
    n = 1 << 14
    ns = unit_vectors(8801, n); wo = unit_vectors(8802, n)
    uv = np.zeros((n, 2), np.float32); xi = uniform_floats(8803, (n, 3))
    ctx, mat = _kernel(cfg)
    wi, pdf, thr = ctx.bsdf_sample(mat, make_isects(wo, ns, ns, uv, mat), xi)
    w64, n64 = wo.astype(np.float64), ns.astype(np.float64)
    c = (w64 * n64).sum(1, keepdims=True)
    refl = 2 * c * n64 - w64
    if cfg["type"] == MIRROR:
        exact = refl
    else:
        eta = np.where(c > 0, 1 / cfg["ior"], cfg["ior"])
        nn = np.where(c > 0, n64, -n64)
        cc = np.abs(c)
        k = 1 - eta ** 2 * (1 - cc ** 2)
        tr = -eta * w64 + (eta * cc - np.sqrt(np.maximum(k, 0))) * nn
        tr /= np.linalg.norm(tr, axis=1, keepdims=True)
        went_back = ((wi.astype(np.float64) * n64).sum(1, keepdims=True) > 0) == (c > 0)
        exact = np.where(went_back, refl, tr)
    sw = R.sample_envelope(cfg, wo, ns, ns, uv, xi)[0]
    with np.errstate(invalid="ignore"):
        inside = ((exact >= sw["lo"] - 1e-6) & (exact <= sw["hi"] + 1e-6)).all(1)
        close = np.abs(wi - exact).max(1) <= 1e-5
    if cfg.get("ior") == 1.0:  # ior = 1, grazing: 1 - |perp|^2 rounds to 0 and the refracted y with it (NON_FINITE_ALLOWED)
        inside |= np.abs(c[:, 0]) < 1e-3
    assert (inside | close).all(), np.where(~(inside | close))[0][:5]
    assert np.isfinite(pdf).all() and (np.isfinite(thr).all() or cfg.get("ior") == 1.0)  # ior = 1: NON_FINITE_ALLOWED


def _reflections_float32(ior, wo_y, xi0):
    """how many of the draws xi0 reflect for wo_y = n.wo (ns = +y): R of the float32 restatement (no libm), xi < R"""
    m = R._M(np.float32)
    inside = wo_y < 0
    eta_i, eta_t = (m.k(ior), m.k(1)) if inside else (m.k(1), m.k(ior))
    refl = R.fresnel(m, np.abs(np.float32(wo_y)), eta_i, eta_t)
    return int((xi0 < refl).sum()), float(refl)


@pytest.mark.parametrize("name", ["glass_10", "glass_10001", "glass_11", "glass_15", "glass_20", "glass_24"])
def test_glass_reflected_fraction_is_fresnel(name):
    """the reflect / refract choice against float64 Fresnel (binomial test at 1e-4 over 2^20 draws per angle) and, exactly, against
    the float32 Fresnel of the restatement; from inside, at the critical angle (the float32 directions nearest it) and beyond, every
    sample reflects where the float32 R is 1, with a finite throughput"""
    cfg = R.ALL_CONFIGS[name]
    ior = float(np.float32(cfg["ior"]))
    ctx, mat = _kernel(cfg)
    n = 1 << 20
    xi = uniform_floats(8804, (n, 3))
    ns = np.tile(np.array([[0, 1, 0]], np.float32), (n, 1)); uv = np.zeros((n, 2), np.float32)
    angles = [0.0, 0.5, 1.0, 1.4, 1.55]
    for th in angles:
        wo = np.tile(np.array([[np.sin(th), np.cos(th), 0]], np.float32), (n, 1))
        wi, pdf, thr = ctx.bsdf_sample(mat, make_isects(wo, ns, ns, uv, mat), xi)
        k = int((wi[:, 1] > 0).sum())
        R64 = float(_fresnel64(np.float64(wo[0, 1]), 1.0, ior))
        p = stats.binomtest(k, n, min(max(R64, 1e-300), 1.0)).pvalue if 0 < R64 < 1 else float(k == round(R64 * n))
        assert p >= 1e-4 / len(angles), (name, th, k / n, R64, p)
        assert k == _reflections_float32(ior, wo[0, 1], xi[:, 0])[0], (name, th)
    if ior <= 1:
        return  # no total internal reflection
    crit = np.arcsin(1 / ior)
    s = np.float32(np.sin(crit))
    near = [np.nextafter(s, np.float32(0)), s, np.nextafter(s, np.float32(1))]
    for sx in near + [np.float32(np.sin(crit + 1e-3)), np.float32(np.sin(crit + 0.3)), np.float32(np.sin(1.5))]:
        wo = np.tile(np.array([[sx, -np.sqrt(1 - np.float64(sx) ** 2), 0]], np.float32), (n, 1))  # inside the medium
        wi, pdf, thr = ctx.bsdf_sample(mat, make_isects(wo, ns, ns, uv, mat), xi)
        k, r32 = _reflections_float32(ior, wo[0, 1], xi[:, 0])
        assert int((wi[:, 1] < 0).sum()) == k, (name, sx)
        if r32 == 1:
            assert (wi[:, 1] < 0).all() and (pdf == 1).all() and np.isfinite(thr).all(), (name, sx)
    # beyond the critical angle R is 1 in float32 as well: the TIR branch is taken for the directions past the nearest one
    assert _reflections_float32(ior, -np.float32(np.cos(crit + 1e-3)), xi[:, 0])[1] == 1.0


# ------------------------------------------------------------------------------------------------ finiteness
# where non-finite outputs are allowed, by name and output:
#   alpha = 0 (test_bsdf_edges_cpu.py::test_alpha_zero_is_pinned): Beckmann's D is 0 / 0 off the horizon, GGX's at wh = n, which the
#   sampler always returns;
#   ior = 1: an index-matched refraction of a grazing wo rounds 1 - |perp|^2 to 0, the refracted y is 0 and the throughput T / 0 = inf
NON_FINITE_ALLOWED = {"beckmann_0": {"f", "pdf", "sample_pdf", "sample_throughput"}, "ggx_0": {"sample_pdf", "sample_throughput"},
                      "glass_10": {"sample_throughput"}}


@pytest.mark.parametrize("name", sorted(R.ALL_CONFIGS))
def test_outputs_finite_wherever_the_restatement_is(name):
    """unit inputs on the sphere: every output the float32 restatement has finite is finite from the kernel, and the restatement's
    own non-finite outputs are the named ones above"""
    cfg = R.ALL_CONFIGS[name]
    n = 1 << 16
    ns = unit_vectors(8811, n); wo = unit_vectors(8812, n); wi = unit_vectors(8813, n)
    ng = ns.copy(); ng[::3] = unit_vectors(8814, len(ng[::3]))
    uv = (uniform_floats(8815, (n, 2)) * np.float32(3) - np.float32(1)).astype(np.float32)
    xi = uniform_floats(8816, (n, 3))
    ctx, mat = _kernel(cfg)
    got = _run(ctx, mat, wo, ng, ns, uv, wi, xi)
    f, pdf = R.bsdf_eval(cfg, wo, ng, ns, uv, wi, "float32")
    swi, spdf, sthr = R.bsdf_sample(cfg, wo, ng, ns, uv, xi, "float32")
    want = dict(f=f, pdf=pdf, sample_wi=swi, sample_pdf=spdf, sample_throughput=sthr)
    allowed = NON_FINITE_ALLOWED.get(name, set())
    for key in want:
        fin_w = np.isfinite(want[key]).reshape(n, -1).all(1)
        fin_g = np.isfinite(got[key]).reshape(n, -1).all(1)
        assert fin_g[fin_w].all(), (name, key, np.where(fin_w & ~fin_g)[0][:5])
        assert (fin_g == fin_w).all() if key in allowed else fin_w.all(), (name, key, np.where(~fin_w)[0][:5])


def test_narrow_lobes_sample_the_mirror_direction():
    """alpha = 1e-4: tan^2 = -alpha^2 log(xi) is below 2^-24 unless xi < 0.0026, cosT = 1 / sqrt(1 + tan^2) rounds to 1 and
    sinT = sqrt(1 - cosT^2) to 0, so the float32 sampler returns wh = n and the sampled direction is Mirror's, bit for bit"""
    n = 1 << 16
    ns = unit_vectors(8821, n); wo = unit_vectors(8822, n)
    d = (wo * ns).sum(1, keepdims=True)
    wo = np.ascontiguousarray(np.where(d < 0, -wo, wo))
    uv = np.zeros((n, 2), np.float32); xi = uniform_floats(8823, (n, 3))
    ctx, mat = _kernel(R.ALL_CONFIGS["beckmann_1e-4"])
    wi, _, _ = ctx.bsdf_sample(mat, make_isects(wo, ns, ns, uv, mat), xi)
    mctx, mmat = _kernel(R.ALL_CONFIGS["mirror"])
    mirror, _, _ = mctx.bsdf_sample(mmat, make_isects(wo, ns, ns, uv, mmat), xi)
    collapsed = -(np.float64(1e-4) ** 2) * np.log(xi[:, 1].astype(np.float64)) < 2.0 ** -25
    same = (wi == mirror).all(1)
    assert same[collapsed].all() and same.mean() > 0.99, (same.mean(), same[collapsed].mean())
