"""Every BSDF of pathed_b200/csrc/shading.cuh restated in numpy, in two modes, plus the tolerance and the inputs that go with it.

mode float64: the same expressions evaluated in double -- the high-precision answer.  Branch thresholds stay the float literals the
    code compares against (0.9999f, 1.6f, 2 pi as a float), so both modes take the same decisions on the same inputs.
mode float32: every operation rounded to float32 in the kernel's order (numpy's float32 arithmetic is IEEE, no FMA), like
    denoise_restatement in tests/test_denoise.py.  A libm step (sin / cos / log / atan / atan2 / acos / tan / exp / pow) takes the
    double-precision value rounded once, which is what the kernel's sinHost / cosHost / logHost / atanHost do.

Followed on purpose: Q10 (Fresnel fixed at 1 -> 1.5, pdf negative for wo.wh < 0), Q11 (no eta^2 on transmission), Q12 (OrenNayar's
back side reports pdf 1), Q13 (Plastic sums both lobes and averages the pdfs), clampf = fminf(hi, fmaxf(v, lo)) (NaN -> lo), the
+-0.9999 axis snap of tfSinPhi, the isinf guards of D / Lambda / G1 and of log(xi) in the Beckmann sampler.

eval_envelope() / sample_envelope(): the float64 results over the inputs moved by +-1 float32 ulp one component at a time (and over
libm results moved by one ulp), widened by the float32 / float64 gap at the tuple itself.  Its width says per tuple how ill-conditioned
an output is.

edge_inputs(): adversarial tuples (grazing, degenerate frames, branch thresholds, random-number boundaries).
EDGE_CONFIGS: parameters outside the reference fixtures' sweep.
"""
import numpy as np

from golden_inputs import (BECKMANN, BSDF_CONFIGS, GGX, GLASS, LAMBERTIAN, MICROFACET, MIRROR, OREN_NAYAR, PLASTIC, make_test_texture,
                           uniform_floats, unit_vectors)

# parameters the reference fixtures do not cover.  alpha = 0 is accepted by ptc_add_material; it is pinned, not changed (see
# tests/test_bsdf_edges.py: NaN D at wh = n)
EDGE_CONFIGS = {
    "beckmann_1e-4": dict(type=MICROFACET, distribution=BECKMANN, alpha=1e-4),
    "beckmann_1": dict(type=MICROFACET, distribution=BECKMANN, alpha=1.0),
    "beckmann_2": dict(type=MICROFACET, distribution=BECKMANN, alpha=2.0),
    "beckmann_0": dict(type=MICROFACET, distribution=BECKMANN, alpha=0.0),
    "ggx_0005": dict(type=MICROFACET, distribution=GGX, alpha=0.005),
    "ggx_002": dict(type=MICROFACET, distribution=GGX, alpha=0.02),
    "ggx_1": dict(type=MICROFACET, distribution=GGX, alpha=1.0),
    "ggx_0": dict(type=MICROFACET, distribution=GGX, alpha=0.0),
    "glass_10": dict(type=GLASS, ior=1.0),
    "glass_10001": dict(type=GLASS, ior=1.0001),
    "glass_24": dict(type=GLASS, ior=2.4),
    "plastic_1e-4": dict(type=PLASTIC, diffuse=(0.3, 0.2, 0.1), distribution=BECKMANN, alpha=1e-4),
}
ALL_CONFIGS = dict(BSDF_CONFIGS, **EDGE_CONFIGS)

SNAP = float(np.float32(0.9999))        # tfSinPhi's axis snap, compared as the float literal
TWO_PI_F = float(np.float32(6.283185307179586))
INV_PI_F = float(np.float32(0.3183098861837907))
PI_F = float(np.float32(np.pi))          # (float)PTC_PI_D, Lambert's divisor


class _M:
    """arithmetic of one mode: casts, libm calls, double-promoted expressions"""

    def __init__(self, dt, libm=0):
        self.dt = dt
        self.libm, self.calls = libm, 0

    def c(self, x):
        return np.asarray(x, self.dt)

    def k(self, x):  # a float literal of the code or a material parameter: a float32 value in both modes
        return np.asarray(np.float32(x), self.dt)

    def lib(self, fn, *a):  # double-precision libm, rounded once in float32 mode
        r = fn(*[np.asarray(x, np.float64) for x in a])
        if self.libm:  # envelope passes: every libm result moved by one float32 ulp, all up / all down / alternating by call
            self.calls += 1
            sign = (1 if self.libm in (1, 3) else -1) * (-1 if self.libm > 2 and self.calls % 2 else 1)
            r = r * (1 + sign * 2.0 ** -23)
        return r.astype(self.dt)

    def dbl(self, x):  # (float)(double expression)
        return np.asarray(x, np.float64).astype(self.dt)


def _v(m, a):
    a = np.asarray(a)
    return m.c(a[..., 0]), m.c(a[..., 1]), m.c(a[..., 2])


def dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def add(a, b):
    return a[0] + b[0], a[1] + b[1], a[2] + b[2]


def sub(a, b):
    return a[0] - b[0], a[1] - b[1], a[2] - b[2]


def scale(a, t):
    return a[0] * t, a[1] * t, a[2] * t


def neg(a):
    return -a[0], -a[1], -a[2]


def cross(a, b):
    return (a[1] * b[2]) - (a[2] * b[1]), (a[2] * b[0]) - (a[0] * b[2]), (a[0] * b[1]) - (a[1] * b[0])


def normalize(a):
    n = np.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
    return a[0] / n, a[1] / n, a[2] / n


def length(a):
    return np.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])


def reflect(w, n):
    return sub(scale(scale(n, dot(w, n)), 2), w)


def where(c, a, b):
    if isinstance(a, tuple):
        return tuple(np.where(c, x, y) for x, y in zip(a, b))
    return np.where(c, a, b)


def clampf(v, lo, hi):
    return np.fmin(hi, np.fmax(v, lo))


def _vec(m, x, y, z, like):
    z0 = np.zeros_like(like)
    return m.k(x) + z0, m.k(y) + z0, m.k(z) + z0


class _Isect:
    def __init__(self, m, wo, ng, ns, uv):
        self.wo, self.n, self.ns = _v(m, wo), _v(m, ng), _v(m, ns)
        uv = np.asarray(uv)
        self.u, self.v = m.c(uv[:, 0]), m.c(uv[:, 1])
        ns_ = self.ns
        same = (ns_[0] == self.wo[0]) & (ns_[1] == self.wo[1]) & (ns_[2] == self.wo[2])
        zero = np.zeros_like(ns_[0])
        xa = where(np.abs(ns_[0]) > np.abs(ns_[1]), normalize((-ns_[2], zero, ns_[0])), normalize((zero, -ns_[2], ns_[1])))
        tx = normalize(cross(ns_, self.wo))
        self.tx = where(same, xa, tx)
        self.tz = where(same, cross(ns_, xa), normalize(cross(ns_, tx)))

    def to_local(self, w):
        return dot(self.tx, w), dot(self.ns, w), dot(self.tz, w)

    def to_world(self, l):
        t, s, z = self.tx, self.ns, self.tz
        return (t[0] * l[0] + s[0] * l[1] + z[0] * l[2], t[1] * l[0] + s[1] * l[1] + z[1] * l[2], t[2] * l[0] + s[2] * l[1] + z[2] * l[2])


# ---------------------------------------------------------------------------------------------------------- tangent frame helpers
def tf_sin(v):
    return np.sqrt(np.fmax(0, 1 - v[1] * v[1]))


def tf_tan2(v):
    return (1 - v[1] * v[1]) / (v[1] * v[1])


def tf_cos_phi(v):
    s = tf_sin(v)
    return np.where(s == 0, 1, clampf(v[0] / s, -1, 1))


def tf_sin_phi(v, snap=SNAP):
    """axis snap: a component at or beyond +-0.9999 replaces v by that axis, in the order x, y, z, -x, -y, -z"""
    x, y, z = v
    one, zero = np.ones_like(x), np.zeros_like(x)
    c = (x, y, z)
    for cond, axis in reversed([(x >= snap, (one, zero, zero)), (y >= snap, (zero, one, zero)), (z >= snap, (zero, zero, one)),
                                (x <= -snap, (-one, zero, zero)), (y <= -snap, (zero, -one, zero)), (z <= -snap, (zero, zero, -one))]):
        c = where(cond, axis, c)
    s = tf_sin(c)
    return np.where(s == 0, 0, clampf(c[2] / s, -1, 1))


def cart_to_sph(m, c):
    phi = m.lib(np.arctan2, c[2], c[0])
    phi = np.where(phi < 0, m.dbl(np.asarray(phi, np.float64) + 2 * np.pi), phi)
    phi = np.where(phi == TWO_PI_F, 0, phi)
    theta = m.lib(np.arccos, clampf(c[1], -1, 1))
    return m.c(phi), theta


def sph_to_cart(m, phi, cos_t, sin_t):
    return sin_t * m.lib(np.cos, phi), cos_t, sin_t * m.lib(np.sin, phi)


# ---------------------------------------------------------------------------------------------------------- material pieces
def albedo(m, cfg, it):
    n = len(it.u)
    if cfg.get("textured"):
        tex = make_test_texture()
        h, w, _ = tex.shape
        u = it.u - np.floor(it.u)
        v = 1 - (it.v - np.floor(it.v))
        fx = np.asarray(u * m.k(w - 1), np.float64); fy = np.asarray(v * m.k(h - 1), np.float64)
        x = np.trunc(fx + np.copysign(0.5, fx)).astype(np.int64); y = np.trunc(fy + np.copysign(0.5, fy)).astype(np.int64)  # roundf
        texel = tex[y, x]
        table = m.lib(np.power, np.arange(256, dtype=np.float32) / np.float32(255), np.float32(2.2))  # c_gammaTable (host powf)
        return tuple(table[texel[:, k]] for k in range(3))
    if "checker" in cfg:
        on, off, res = cfg["checker"]
        ui = np.floor(it.u * m.k(res[0])).astype(np.int64); vi = np.floor(it.v * m.k(res[1])).astype(np.int64)
        pick = np.fmod(ui, 2) == np.fmod(vi, 2)  # C remainder: sign of the dividend
        return tuple(np.where(pick, m.k(on[k]), m.k(off[k])) for k in range(3))
    d = cfg.get("diffuse", (0, 0, 0))
    return tuple(m.k(d[k]) + np.zeros(n, m.dt) for k in range(3))


def fresnel(m, cos_i, eta_i, eta_t):
    sin_t = (eta_i / eta_t) * np.sqrt(np.fmax(0, 1 - cos_i * cos_i))
    cos_t = np.sqrt(np.fmax(0, 1 - sin_t * sin_t))
    r_par = (eta_t * cos_i - eta_i * cos_t) / (eta_t * cos_i + eta_i * cos_t)
    r_perp = (eta_i * cos_i - eta_t * cos_t) / (eta_i * cos_i + eta_t * cos_t)
    return np.where(sin_t > 1, 1, 0.5 * (r_par * r_par + r_perp * r_perp))


def mf_d(m, cfg, wh, snap=SNAP):
    alpha = m.k(cfg["alpha"])
    alpha2 = alpha * alpha
    tan2 = tf_tan2(wh)
    cos2 = wh[1] * wh[1]
    cos4 = cos2 * cos2
    if cfg["distribution"] == BECKMANN:
        cp, sp = tf_cos_phi(wh), tf_sin_phi(wh, snap)
        num = m.lib(np.exp, -tan2 * (cp * cp / alpha2 + sp * sp / alpha2))
        den = m.dbl(np.pi * np.float64(alpha2) * np.asarray(cos4, np.float64))
        d = num / den
    else:
        s = alpha2 + tan2
        d = alpha2 / m.dbl(np.pi * np.asarray(cos4, np.float64) * np.asarray(s, np.float64) * np.asarray(s, np.float64))
    return np.where(np.isinf(tan2), 0, d)


def mf_pdf(m, cfg, wh, snap=SNAP):
    return mf_d(m, cfg, wh, snap) * np.abs(wh[1])


def beckmann_lambda(m, alpha, w):
    abs_tan = np.abs(tf_sin(w) / w[1])
    cp, sp = tf_cos_phi(w), tf_sin_phi(w)
    a_ = np.sqrt((cp * cp) * alpha * alpha + (sp * sp) * alpha * alpha)
    a = 1 / (a_ * abs_tan)
    lam = (1 - m.k(1.259) * a + m.k(0.396) * a * a) / (m.k(3.535) * a + m.k(2.181) * a * a)
    return np.where(np.isinf(abs_tan) | (a >= m.k(1.6)), 0, lam)


def ggx_g1(m, alpha, v):
    tan2 = tf_tan2(v)
    s = 1 + alpha * alpha * tan2
    return np.where(np.isinf(tan2), 0, 2 / (1 + np.sqrt(s)))


def mf_g(m, cfg, wo, wi):
    alpha = m.k(cfg["alpha"])
    if cfg["distribution"] == BECKMANN:
        return 1 / (1 + beckmann_lambda(m, alpha, wo) + beckmann_lambda(m, alpha, wi))
    return ggx_g1(m, alpha, wo) * ggx_g1(m, alpha, wi)


def lambert_f(m, cfg, it, wiw):
    rej = (dot(it.wo, it.ns) < 0) | (dot(wiw, it.ns) < 0)
    wi = normalize(it.to_local(wiw))
    pdf = np.where(rej, 0, wi[1] * m.k(INV_PI_F))
    a = albedo(m, cfg, it)
    f = tuple(np.where(rej, 0, x / m.k(PI_F)) for x in a)
    return f, pdf


def microfacet_f(m, cfg, it, wiw, snap=SNAP):
    rej = (dot(it.wo, it.ns) < 0) | (dot(wiw, it.ns) < 0)
    wo, wi = normalize(it.to_local(it.wo)), normalize(it.to_local(wiw))
    cos_o, cos_i = np.abs(wo[1]), np.abs(wi[1])
    wh = normalize(add(wo, wi))
    pdf = mf_pdf(m, cfg, wh, snap) / (4 * dot(wo, wh))
    zero = (cos_o == 0) | (cos_i == 0) | ((wh[0] == 0) & (wh[1] == 0) & (wh[2] == 0))
    F = fresnel(m, clampf(dot(wi, wh), 0, 1), m.k(1), m.k(1.5))  # Q10
    D = mf_d(m, cfg, wh, snap)
    G = mf_g(m, cfg, wo, wi)
    val = (1 * D) * G * F / (4 * cos_i * cos_o)
    val = np.where(rej | zero, 0, val)
    return (val, val, val), np.where(rej, 0, pdf)


def oren_nayar_ab(m, sigma):
    """A and B as ptc_add_material computes them, in float32 (material parameters)"""
    s = np.float32(sigma)
    s2 = s * s
    return m.k(1 - (s2 / (2 * (s2 + np.float32(0.33))))), m.k((np.float32(0.45) * s2) / (s2 + np.float32(0.09)))


def oren_nayar_f(m, cfg, it, wiw):
    A, B = oren_nayar_ab(m, cfg.get("sigma", 0.0))
    back = (dot(it.n, it.wo) < 0) | (dot(it.ns, it.wo) < 0)
    lwo, lwi = normalize(it.to_local(it.wo)), normalize(it.to_local(wiw))
    below = back | (lwo[1] < 0) | (lwi[1] < 0)
    phi_i, th_i = cart_to_sph(m, lwi)
    phi_o, th_o = cart_to_sph(m, lwo)
    alpha, beta = np.fmax(th_i, th_o), np.fmin(th_i, th_o)
    pdf = np.where(below, 1, lwi[1] * m.k(INV_PI_F))  # Q12
    thr = m.k(INV_PI_F) * (A + B * np.fmax(0, m.lib(np.cos, phi_i - phi_o)) * m.lib(np.sin, alpha) * m.lib(np.tan, beta))
    d = cfg["diffuse"]
    return tuple(np.where(below, 0, m.k(d[k]) * thr) for k in range(3)), pdf


def _eval(m, cfg, it, wiw, snap=SNAP):
    t = cfg["type"]
    if t == LAMBERTIAN:
        return lambert_f(m, cfg, it, wiw)
    if t == OREN_NAYAR:
        return oren_nayar_f(m, cfg, it, wiw)
    if t == MICROFACET:
        return microfacet_f(m, cfg, it, wiw, snap)
    if t == PLASTIC:
        fl, pl = lambert_f(m, cfg, it, wiw)
        fm, pm = microfacet_f(m, cfg, it, wiw, snap)
        return add(fl, fm), (pl + pm) / 2
    z = np.zeros_like(it.u)
    return (z, z, z), z  # Mirror, Glass


def cosine_sample(m, x1, x2):
    rad = np.sqrt(x1)
    phi = m.dbl(2 * np.pi * np.asarray(x2, np.float64))
    return rad * m.lib(np.cos, phi), np.sqrt(1 - x1), rad * m.lib(np.sin, phi)


def mf_sample_wh(m, cfg, x1, x2):
    alpha = m.k(cfg["alpha"])
    if cfg["distribution"] == BECKMANN:
        phi = m.dbl(np.asarray(x1, np.float64) * np.pi * 2.0)
        log_xi = m.lib(np.log, x2)
        log_xi = np.where(np.isinf(log_xi), 0, log_xi)
        tan2 = -alpha * alpha * log_xi
        cos_t = 1 / np.sqrt(1 + tan2)
        sin_t = np.sqrt(np.fmax(0, 1 - cos_t * cos_t))
        return sph_to_cart(m, phi, cos_t, sin_t)
    theta = m.lib(np.arctan, (alpha * np.sqrt(x1)) / np.sqrt(1 - x1))
    phi = m.k(TWO_PI_F) * x2
    return sph_to_cart(m, phi, m.lib(np.cos, theta), m.lib(np.sin, theta))


def _sample(m, cfg, it, xi):
    x0, x1, x2 = m.c(xi[:, 0]), m.c(xi[:, 1]), m.c(xi[:, 2])
    t = cfg["type"]
    ey = _vec(m, 0, 1, 0, it.u)
    if t in (LAMBERTIAN, OREN_NAYAR):
        l = cosine_sample(m, x0, x1)
        wi = it.to_world(l)
        f, _ = _eval(m, cfg, it, wi)
        return wi, l[1] * m.k(INV_PI_F), f
    if t == MIRROR:
        lwi = reflect(it.to_local(it.wo), ey)
        tt = np.fmax(0, 1 / lwi[1])
        return it.to_world(lwi), np.ones_like(tt), (tt, tt, tt)
    if t == GLASS:
        lwo = it.to_local(it.wo)
        inside = lwo[1] < 0
        ior = m.k(cfg["ior"]) + np.zeros_like(it.u)
        eta_i, eta_t = np.where(inside, ior, m.k(1)), np.where(inside, m.k(1), ior)
        normal = where(inside, scale(ey, -1), ey)
        inc_perp = sub(lwo, scale(normal, dot(lwo, normal)))
        trans_perp = scale(neg(inc_perp), eta_i / eta_t)
        perp_len2 = length(trans_perp) * length(trans_perp)
        trans_par = scale(normal, -np.sqrt(np.fmax(0, 1 - perp_len2)))
        refracted = normalize(add(trans_par, trans_perp))
        R = fresnel(m, np.abs(lwo[1]), eta_i, eta_t)
        lwi = reflect(lwo, ey)
        refl = x0 < R
        T = 1 - R
        tt = np.where(refl, R / np.abs(lwi[1]), T / np.abs(refracted[1]))
        return it.to_world(where(refl, lwi, refracted)), np.where(refl, R, T), (tt, tt, tt)
    if t == MICROFACET:
        wo = it.to_local(it.wo)
        wh = mf_sample_wh(m, cfg, x0, x1)
        wi = it.to_world(reflect(wo, wh))
        pdf = mf_pdf(m, cfg, wh) / (4 * dot(wo, wh))
        f, _ = microfacet_f(m, cfg, it, wi)
        return wi, pdf, f
    # Plastic: xi0 > 0.5 picks the diffuse lobe
    diffuse = x0 > m.k(0.5)
    l = cosine_sample(m, x1, x2)
    wi_d = it.to_world(l)
    wo = it.to_local(it.wo)
    wh = mf_sample_wh(m, cfg, x1, x2)
    wi_s = it.to_world(reflect(wo, wh))
    wi = where(diffuse, wi_d, wi_s)
    sampled = np.where(diffuse, l[1] * m.k(INV_PI_F), mf_pdf(m, cfg, wh) / (4 * dot(wo, wh)))
    fl, pl = lambert_f(m, cfg, it, wi)
    fm, pm = microfacet_f(m, cfg, it, wi)
    return wi, (sampled + np.where(diffuse, pm, pl)) / 2, add(fl, fm)


def _stack(v):
    return np.stack(v, -1)


def bsdf_eval(cfg, wo, ng, ns, uv, wi, mode="float64", snap=SNAP, libm=0):
    """(f (n, 3), pdf (n,)) of Material::f"""
    m = _M(np.float64 if mode == "float64" else np.float32, libm)
    with np.errstate(all="ignore"):
        it = _Isect(m, wo, ng, ns, uv)
        f, pdf = _eval(m, cfg, it, _v(m, wi), snap)
        n = len(it.u)
        return _stack(f) + np.zeros((n, 3), m.dt), np.asarray(pdf, m.dt) + np.zeros(n, m.dt)


def bsdf_sample(cfg, wo, ng, ns, uv, xi, mode="float64", libm=0):
    """(wi (n, 3), pdf (n,), throughput (n, 3)) of Material::sample with the three replayed random numbers"""
    m = _M(np.float64 if mode == "float64" else np.float32, libm)
    with np.errstate(all="ignore"):
        it = _Isect(m, wo, ng, ns, uv)
        wi, pdf, thr = _sample(m, cfg, it, np.asarray(xi))
        n = len(it.u)
        return _stack(wi) + np.zeros((n, 3), m.dt), np.asarray(pdf, m.dt) + np.zeros(n, m.dt), _stack(thr) + np.zeros((n, 3), m.dt)


# ---------------------------------------------------------------------------------------------------------- envelope
def _ulp_moves(arrays, clip01):
    """yield (input arrays with one float32 component moved by one ulp up or down, 0), then (the inputs, libm pass 1..4)"""
    for libm in (1, 2, 3, 4):
        yield list(arrays), libm
    for k, a in enumerate(arrays):
        if clip01[k] is None:
            continue
        for c in range(a.shape[1]):
            for direction in (np.inf, -np.inf):
                b = a.copy()
                b[:, c] = np.nextafter(a[:, c], np.float32(direction))
                if clip01[k]:
                    b[:, c] = np.clip(b[:, c], np.float32(0), np.float32(1 - 2.0 ** -24))
                out = list(arrays)
                out[k] = b
                yield out, 0


def _envelope(fn, arrays, clip01):
    center64 = [np.asarray(x, np.float64) for x in fn(*arrays, mode="float64")]
    center32 = [np.asarray(x, np.float64) for x in fn(*arrays, mode="float32")]
    lo = [c.copy() for c in center64]
    hi = [c.copy() for c in center64]
    with np.errstate(invalid="ignore"):
        for moved, libm in _ulp_moves(arrays, clip01):
            for k, r in enumerate(fn(*moved, mode="float64", libm=libm)):
                r = np.asarray(r, np.float64)
                lo[k] = np.fmin(lo[k], r)
                hi[k] = np.fmax(hi[k], r)
        out = []
        for c64, c32, l, h in zip(center64, center32, lo, hi):
            gap = np.abs(c32 - c64)
            gap = np.where(np.isnan(gap), 0, gap)
            # a few float32 ulp more for the libm steps a device library rounds differently (libdevice expf / atan2f / acosf / tanf)
            slack = 4 * np.spacing(np.abs(c32).astype(np.float32)).astype(np.float64)
            slack = np.where(np.isfinite(slack), slack, 0)
            lo_, hi_ = np.fmin(l - gap, c32), np.fmax(h + gap, c32)  # c32 itself: l - gap cancels when gap ~ l
            out.append(dict(f64=c64, f32=c32, lo=lo_ - slack, hi=hi_ + slack, width=hi_ - lo_))
    return out


def eval_envelope(cfg, wo, ng, ns, uv, wi):
    """[f, pdf] as dicts of f64 / f32 / lo / hi arrays"""
    def fn(wo, ng, ns, wi, mode, libm=0):
        return bsdf_eval(cfg, wo, ng, ns, uv, wi, mode, libm=libm)
    return _envelope(fn, [wo, ng, ns, wi], [False, False, False, False])


def sample_envelope(cfg, wo, ng, ns, uv, xi):
    """[wi, pdf, throughput] as dicts of f64 / f32 / lo / hi arrays"""
    def fn(wo, ng, ns, xi, mode, libm=0):
        return bsdf_sample(cfg, wo, ng, ns, uv, xi, mode, libm=libm)
    return _envelope(fn, [wo, ng, ns, xi], [False, False, False, True])


def envelope_ulps(env):
    """width of the input-perturbation envelope (libm slack not counted) in float32 ulps of the float64 value, per tuple (the largest
    component for vectors); inf where it is not finite.  Values below 1e-6 are measured in ulps of 1e-6, the floor of rel_err."""
    with np.errstate(invalid="ignore", over="ignore"):
        ref = np.abs(env["f64"])
        if ref.ndim > 1:
            ref = np.broadcast_to(np.max(np.where(np.isfinite(ref), ref, 0), -1, keepdims=True), ref.shape)
        ulp = np.spacing(np.maximum(ref, 1e-6).astype(np.float32)).astype(np.float64)
        w = env["width"] / ulp
        w = np.where(np.isfinite(w), w, np.inf)
    return w.max(-1) if w.ndim > 1 else w


def _sign_class(x):
    """-1 / 0 / +1 for finite values, 2 for NaN, +-3 for +-inf"""
    x = np.asarray(x, np.float64)
    with np.errstate(invalid="ignore"):
        return np.where(np.isnan(x), 2, np.where(np.isinf(x), 3 * np.sign(x), np.sign(x))).astype(np.int8)


def judge(cfg, inputs, got, rel=1e-5, well_ulps=10):
    """Checks an implementation's eval / sample outputs (got: f, pdf, sample_wi, sample_pdf, sample_throughput) on inputs
    (wo, ng, ns, uv, wi, xi) against the restatement:
      (a) finite / NaN / inf pattern and sign of every output equal to the float32 restatement's,
      (b) outputs whose envelope is narrower than well_ulps float32 ulps within rel of the float64 restatement,
      (c) every other finite output inside the envelope.
    The sampled throughput of a non-delta BSDF is judged as f of the restatement at the implementation's OWN sampled direction (the sampled direction is
    ill-conditioned in the last bit of libm; f at a given direction is not).  Returns {output: [(tuple, reason), ...]} of failures."""
    from parity import rel_err
    wo, ng, ns, uv, wi, xi = inputs
    ef, ep = eval_envelope(cfg, wo, ng, ns, uv, wi)
    sw, sp, st = sample_envelope(cfg, wo, ng, ns, uv, xi)
    if cfg["type"] not in (MIRROR, GLASS):  # delta BSDFs: f is 0, the throughput is judged with the sample itself
        st, _ = eval_envelope(cfg, wo, ng, ns, uv, np.ascontiguousarray(got["sample_wi"], np.float32))
    fails = {}
    for key, env in (("f", ef), ("pdf", ep), ("sample_wi", sw), ("sample_pdf", sp), ("sample_throughput", st)):
        g = np.asarray(got[key], np.float64)
        bad = []
        pat = _sign_class(g) != _sign_class(env["f32"])
        pat = pat.any(-1) if pat.ndim > 1 else pat
        for k in np.where(pat)[0]:
            bad.append((int(k), "pattern/sign: got %r, float32 restatement %r" % (g[k], env["f32"][k])))
        well = envelope_ulps(env) < well_ulps
        with np.errstate(invalid="ignore"):
            e = rel_err(g, env["f64"])
            e = e.max(-1) if e.ndim > 1 else e
            off = well & ~pat & (e > rel)
            for k in np.where(off)[0]:
                bad.append((int(k), "well-conditioned, rel err %.3g vs float64" % e[k]))
            out = np.isfinite(g) & ((g < env["lo"]) | (g > env["hi"]))
            out = out.any(-1) if out.ndim > 1 else out
            for k in np.where(out & ~pat & ~off)[0]:
                bad.append((int(k), "outside envelope: got %r, [%r, %r]" % (g[k], env["lo"][k], env["hi"][k])))
        if bad:
            fails[key] = bad
    return fails


# ---------------------------------------------------------------------------------------------------------- adversarial tuples
def _f32(x):
    return np.asarray(x, np.float32)


def _unit(v):
    v = np.asarray(v, np.float64)
    return _f32(v / np.linalg.norm(v, axis=-1, keepdims=True))


def _rot_y_to(n):
    """rotation (float64, rows) taking +y to the unit vector n"""
    n = np.asarray(n, np.float64)
    a = np.array([1.0, 0, 0]) if abs(n[0]) < 0.9 else np.array([0, 0, 1.0])
    t = np.cross(n, a); t /= np.linalg.norm(t)
    b = np.cross(t, n)
    return np.stack([t, n, b], 1)  # columns: x, y, z axes


def _dir(theta, phi):
    return np.stack([np.sin(theta) * np.cos(phi), np.cos(theta), np.sin(theta) * np.sin(phi)], -1)


def edge_inputs(cfg):
    """(wo, ng, ns, uv, wi, xi, tags): every case of the issue list, each tagged with what it exercises.  Normals are the axes,
    a few tilted unit vectors and a vector whose y is exactly the 0.9999 snap threshold; directions are placed in the frame of the
    shading normal and rounded to float32."""
    rows, tags = [], []

    def add(tag, wo, ns, wi, xi, ng=None):
        rows.append((_f32(wo), _f32(ns if ng is None else ng), _f32(ns), _f32(wi), _f32(xi)))
        tags.append(tag)

    one = np.float32(1)
    tiny = [0.0, float(np.float32(2.0 ** -149)), float(np.float32(1e-7)), float(np.spacing(np.float32(0))), -float(np.float32(2.0 ** -149)), -1e-7]
    snap = np.float32(SNAP)
    near_snap = [float(np.nextafter(snap, np.float32(-1))), float(snap), float(np.nextafter(snap, one))]
    normals = [np.array(n, np.float32) for n in ([0, 1, 0], [0, -1, 0], [1, 0, 0], [0, 0, 1], [0, 0, -1])]
    normals += [_unit([0.3, 0.9, -0.2]), _unit([-0.6, 0.1, 0.78]), _unit([0.0, 1.0, 1e-3])]
    xis = [(0.5, 0.5, 0.5), (0.0, 0.0, 0.0), (0.0, 0.5, 0.25), (0.25, 0.0, 0.0), (1 - 2.0 ** -24, 1 - 2.0 ** -24, 1 - 2.0 ** -24),
           (0.5 - 2.0 ** -24, 0.3, 0.7), (0.5 + 2.0 ** -24, 0.3, 0.7), (0.5, 0.3, 0.7), (0.7, 2.0 ** -24, 0.9), (0.3, 0.9, 2.0 ** -24)]

    for ni, ns in enumerate(normals):
        R = _rot_y_to(ns)
        to_w = lambda l: _unit(np.asarray(l, np.float64) @ R.T)
        for xi in xis:
            # wo exactly along ns (wh = ns, tan^2 = 0 for the mirror wi), wo = -ns, wi = -wo
            add("wo=ns", ns, ns, ns, xi)
            add("wo=-ns", -ns, ns, ns, xi)
            add("wi=-wo", to_w(_dir(0.7, 1.1)), ns, -to_w(_dir(0.7, 1.1)), xi)
            for th in (0.0, 0.3, 1.2, 1.5707):
                wo = to_w(_dir(th, 0.4))
                add("mirror wi", wo, ns, _unit(2 * np.dot(wo, ns) * ns.astype(np.float64) - wo), xi)
        # grazing: n.w of 0, +-1 ulp, 1e-7 (directions built exactly in the local frame of an axis normal, tilted ones rounded)
        for c in tiny:
            s = np.sqrt(max(0.0, 1 - c * c))
            g = to_w([s, c, 0.0]) if ni >= 5 else _f32(np.asarray([s, c, 0.0]) @ R.T)
            for xi in xis[:4]:
                add("grazing wo", g, ns, to_w(_dir(0.5, 2.0)), xi)
                add("grazing wi", to_w(_dir(0.5, 2.0)), ns, g, xi)
                add("grazing both", g, ns, _f32(np.asarray([-s, c, 0.0]) @ R.T), xi)
        # angles around the critical angle of glass (both sides) and total internal reflection
        if cfg["type"] == GLASS and cfg["ior"] > 1:
            crit = np.arcsin(1 / cfg["ior"])
            for th in (crit - 1e-6, crit, crit + 1e-6, crit + 0.2, 1.4):
                for xi0 in (0.0, 0.5, 1 - 2.0 ** -24):
                    inside = to_w(_dir(np.pi - th, 0.3))
                    add("glass inside", inside, ns, ns, (xi0, 0.5, 0.5))
        # Fresnel reflectance R as the random number: the reflect / refract choice at xi = R exactly and one ulp either side
        if cfg["type"] == GLASS:
            for th in (0.2, 1.0, 1.5):
                wo = to_w(_dir(th, 0.1))
                m = _M(np.float32)
                with np.errstate(all="ignore"):
                    it = _Isect(m, wo[None], ns[None], ns[None], np.zeros((1, 2), np.float32))
                    lwo = it.to_local(it.wo)
                    refl = float(fresnel(m, np.abs(lwo[1]), m.k(1), m.k(cfg["ior"]))[0])
                for x0 in (np.nextafter(np.float32(refl), np.float32(0)), refl, np.nextafter(np.float32(refl), one)):
                    add("xi=R", wo, ns, ns, (x0, 0.5, 0.5))
    # ns != ng with dot products of opposite sign (OrenNayar back side, Q12), rejection on one normal but not the other
    for k, (th_o, th_i) in enumerate([(1.4, 0.5), (0.3, 1.5), (1.55, 1.55), (0.9, 0.2)]):
        ns = normals[5]
        R = _rot_y_to(ns)
        ng = _unit(R @ np.array([np.sin(0.5), np.cos(0.5), 0.0]))
        wo = _unit(R @ _dir(th_o, np.pi))  # tilted away from ng: ng.wo < 0 < ns.wo for the grazing ones
        for xi in xis[:3]:
            add("ns!=ng", wo, ns, _unit(R @ _dir(th_i, 0.3)), xi, ng=ng)
            add("ns!=ng flipped", wo, ns, _unit(R @ _dir(th_i, 0.3)), xi, ng=_f32(-ng))
    # the axis snap at +-0.9999: half vectors and directions with one component at, and one ulp either side of, the threshold.
    # wo = wi = v makes wh = v exactly (up to rounding) and exercises tfSinPhi / tfCosPhi in D, Lambda and G1
    ns = normals[0]
    for c in near_snap:
        for axis in range(3):
            for sign in (1, -1):
                rest = np.sqrt(max(0.0, 1 - c * c))
                v = np.zeros(3); v[axis] = sign * c; v[(axis + 1) % 3] = rest * 0.6; v[(axis + 2) % 3] = rest * 0.8
                v = _f32(v)
                v[axis] = np.float32(sign * c)
                if v[1] < 0:
                    v = _f32([v[0], -v[1], v[2]])
                for xi in xis[:2]:
                    add("snap", v, ns, v, xi)
                    add("snap wi", _f32(_dir(0.3, 0.2)), ns, v, xi)
        # shading normal with y at the threshold: the frame, and tfSinPhi of the local vectors
        nsn = _f32([np.sqrt(max(0.0, 1 - c * c)), c, 0.0])
        add("snap ns", nsn, nsn, nsn, xis[0])
    # wh exactly along y: s == 0 branches of tfCosPhi / tfSinPhi
    add("s=0", _f32([0, 1, 0]), _f32([0, 1, 0]), _f32([0, 1, 0]), xis[0])
    # wo within 1e-23 of an axis normal but not equal to it: |cross(ns, wo)|^2 underflows, makeFrame divides by 0 and the tangent axes
    # are NaN / inf.  Every local vector is then NaN, and clampf's NaN -> lo (fmaxf drops the NaN) is what keeps cartToSph's theta = pi
    # and Oren-Nayar's f finite: the one place bsdf_eval / bsdf_sample observe clampf's NaN semantics
    for t in (1e-23, 2.0 ** -80, 1e-30):
        for wo_, ns_ in (((t, 1, 0), (0, 1, 0)), ((0, t, 1), (0, 0, 1)), ((-1, 0, t), (-1, 0, 0)), ((t, -1, -t), (0, -1, 0))):
            for wi_ in ((0.3, 0.8, 0.52), (0, 1, 0), ns_):
                add("near-normal wo", _f32(wo_), _f32(ns_), _f32(wi_), xis[0])
    # Beckmann: a = 1 / (alpha tan) around the 1.6 threshold, for this config's alpha
    if cfg.get("alpha", 0) > 0:
        for a in (1.6 * (1 - 1e-6), 1.6, 1.6 * (1 + 1e-6), 0.5, 3.0):
            th = np.arctan(1 / (a * cfg["alpha"]))
            for phi in (0.0, 0.7):
                w = _f32(_dir(th, phi))
                add("lambda a=1.6", w, _f32([0, 1, 0]), _f32(_dir(0.3, phi + 2.0)), xis[0])
    # random-number boundaries everywhere on generic geometry
    R = _rot_y_to(normals[5])
    for xi in xis + [(0.0, 1 - 2.0 ** -24, 0.0), (1 - 2.0 ** -24, 0.0, 1 - 2.0 ** -24), (2.0 ** -24, 2.0 ** -24, 2.0 ** -24)]:
        for th in (0.0, 0.6, 1.3, 1.5706):
            add("xi edge", _unit(R @ _dir(th, 0.9)), normals[5], _unit(R @ _dir(0.4, 2.5)), xi)
    # random unit tuples on the sphere (back sides included) and near the mirror direction, as the fixtures have
    n_rand = 512
    ns = unit_vectors(9101, n_rand); wo = unit_vectors(9102, n_rand); wi = unit_vectors(9103, n_rand)
    d = (wo * ns).sum(1, keepdims=True)
    wi[n_rand // 2:] = _unit(2 * d[n_rand // 2:] * ns[n_rand // 2:] - wo[n_rand // 2:] + 0.003 * unit_vectors(9104, n_rand - n_rand // 2))
    xi = uniform_floats(9105, (n_rand, 3))
    for k in range(n_rand):
        add("random", wo[k], ns[k], wi[k], xi[k])
    wo, ng, ns, wi, xi = (np.ascontiguousarray(np.stack([r[j] for r in rows])) for j in range(5))
    uv = np.ascontiguousarray((uniform_floats(9106, (len(wo), 2)) * np.float32(1.5) - np.float32(0.25)).astype(np.float32))
    return wo, ng, ns, uv, wi, xi, np.array(tags)


# ---------------------------------------------------------------------------------------------------------- quadrature in half-vector space
# Every direction wi != -wo is reflect(wo, wh) for exactly one half vector wh with wo.wh > 0, and dw_i = 4 |wo.wh| dw_h.  Half vectors
# are parametrised by s = ln(tan(theta_h) / w) and phi_h (w: the lobe's width, alpha for the microfacet family, 1 for the diffuse ones), so
# one grid resolves a lobe of any width and the diffuse part of Plastic alike.  The local frame is y-up; wo lies in the xy plane.
def halfvector_coords(wo_l, wi_l, w):
    """(s, phi_h) of the half vector of local directions (float64 arrays (n, 3))"""
    wh = np.asarray(wo_l, np.float64) + np.asarray(wi_l, np.float64)
    with np.errstate(all="ignore"):
        t = np.hypot(wh[:, 0], wh[:, 2]) / wh[:, 1]
        s = np.log(t / w)
    return s, np.mod(np.arctan2(wh[:, 2], wh[:, 0]), 2 * np.pi)


def halfvector_nodes(s_edges, phi_edges, wo_l, w, order=6, return_wh=False):
    """Gauss-Legendre nodes of every (s, phi) cell: (wi_local (cells, k, 3), weight (cells, k)) with weight = dw_i of the node; with
    return_wh also (wh_local, dw_h) of the nodes"""
    x, g = np.polynomial.legendre.leggauss(order)
    s0, s1 = s_edges[:-1], s_edges[1:]
    p0, p1 = phi_edges[:-1], phi_edges[1:]
    S = (s0[:, None] + (s1 - s0)[:, None] * (x[None, :] + 1) / 2)            # (ns, order)
    Ws = (s1 - s0)[:, None] * g[None, :] / 2
    P = (p0[:, None] + (p1 - p0)[:, None] * (x[None, :] + 1) / 2)
    Wp = (p1 - p0)[:, None] * g[None, :] / 2
    ss = S[:, None, :, None] + 0 * P[None, :, None, :]
    pp = P[None, :, None, :] + 0 * S[:, None, :, None]
    ww = Ws[:, None, :, None] * Wp[None, :, None, :]
    ss, pp, ww = ss.reshape(len(s0) * len(p0), -1), pp.reshape(len(s0) * len(p0), -1), ww.reshape(len(s0) * len(p0), -1)
    rho = np.exp(ss) * w                                                       # tan(theta_h)
    cos_h = 1 / np.sqrt(1 + rho * rho)
    wh = np.stack([rho * cos_h * np.cos(pp), cos_h, rho * cos_h * np.sin(pp)], -1)
    wo = np.asarray(wo_l, np.float64)
    d = (wh * wo).sum(-1)
    wi = 2 * d[..., None] * wh - wo
    # dw_h = sin(theta_h) dtheta_h dphi = rho cos^3 drho dphi, drho = rho ds
    dwh = ww * rho * rho * cos_h ** 3
    if return_wh:
        return wi, dwh * 4 * np.abs(d), wh, dwh
    return wi, dwh * 4 * np.abs(d)


def local_frame_isect(theta_o, tilt_ng=0.0):
    """wo at theta_o from ns = +y in the xy plane (float32), ng = ns or ns tilted by tilt_ng about z; makeFrame(ns, wo) then has
    tx = -z, ns = y, tz = x.  Returns (wo, ng, ns) as (1, 3) float32 arrays"""
    wo = np.array([[np.sin(theta_o), np.cos(theta_o), 0.0]], np.float32)
    ns = np.array([[0.0, 1.0, 0.0]], np.float32)
    ng = np.array([[np.sin(tilt_ng), np.cos(tilt_ng), 0.0]], np.float32) if tilt_ng else ns
    return wo, ng, ns


def frame_of(wo, ns):
    """the float64 frame makeFrame(ns, wo) builds, as rows tx, ns, tz"""
    wo = np.asarray(wo, np.float64)[0]; ns = np.asarray(ns, np.float64)[0]
    if (wo == ns).all():
        xa = np.array([-ns[2], 0, ns[0]]) if abs(ns[0]) > abs(ns[1]) else np.array([0, -ns[2], ns[1]])
        xa /= np.linalg.norm(xa)
        return np.stack([xa, ns, np.cross(ns, xa)])
    tx = np.cross(ns, wo); tx /= np.linalg.norm(tx)
    tz = np.cross(ns, tx); tz /= np.linalg.norm(tz)
    return np.stack([tx, ns, tz])


def lobe_width(cfg):
    return max(cfg.get("alpha", 1.0), 1e-30) if cfg["type"] in (MICROFACET, PLASTIC) else 1.0


def halfvector_grid(cfg, theta_o, tilt_ng=0.0, n_s=160, n_phi=48, order=4, return_wh=False):
    """(wo, ng, ns, frame, s_edges, phi_edges, wi_world (cells, k, 3) float32, weight (cells, k)): quadrature nodes covering every
    direction, s from ln(1e-6) to ln(1e5 / w); with return_wh the local half vectors and their dw_h follow"""
    wo, ng, ns = local_frame_isect(theta_o, tilt_ng)
    F = frame_of(wo, ns)
    w = lobe_width(cfg)
    se = np.linspace(np.log(1e-6), np.log(1e5 / w), n_s + 1)
    pe = np.linspace(0, 2 * np.pi, n_phi + 1)
    wi_l, wt, wh, dwh = halfvector_nodes(se, pe, F @ wo[0].astype(np.float64), w, order, return_wh=True)
    out = (wo, ng, ns, F, se, pe, np.asarray(wi_l @ F, np.float32), wt)
    return out + (wh, dwh) if return_wh else out


def upper_pdf_integral(cfg, theta_o, snap=SNAP, tilt_ng=0.0, evaluate=None):
    """integral of pdf over the directions above the shading surface.  evaluate(wo, ng, ns, uv, wi) -> pdf replaces the restatement
    (float64) when given"""
    wo, ng, ns, F, se, pe, wi, wt = halfvector_grid(cfg, theta_o, tilt_ng)
    wi, wt = wi.reshape(-1, 3), wt.reshape(-1)
    n = len(wi)
    args = (np.repeat(wo, n, 0), np.repeat(ng, n, 0), np.repeat(ns, n, 0), np.zeros((n, 2), np.float32), wi)
    pdf = evaluate(*args) if evaluate else bsdf_eval(cfg, *args, "float64", snap=snap)[1]
    above = (wi.astype(np.float64) @ ns[0].astype(np.float64)) >= 0
    return float(np.where(above, pdf, 0) @ wt)


def halfvector_cell_nodes(s0, s1, p0, p1, wo_l, w, order=4, sub=1):
    """quadrature nodes of the (s, phi) cells [s0, s1] x [p0, p1] (arrays of m cells), each cut into sub x sub pieces:
    (wi_local (m, k, 3), dw_i (m, k), wh_local (m, k, 3), dw_h (m, k)), k = (sub * order)^2"""
    m = len(s0)
    f = (np.arange(sub + 1) / sub)
    se = s0[:, None] + (s1 - s0)[:, None] * f[None, :]                       # (m, sub + 1)
    pe = p0[:, None] + (p1 - p0)[:, None] * f[None, :]
    out = []
    for a in range(sub):
        for b in range(sub):
            out.append(halfvector_nodes_cells(se[:, a], se[:, a + 1], pe[:, b], pe[:, b + 1], wo_l, w, order))
    return tuple(np.concatenate([o[j] for o in out], 1) for j in range(4)) if m else None


def halfvector_nodes_cells(s0, s1, p0, p1, wo_l, w, order):
    x, g = np.polynomial.legendre.leggauss(order)
    S = s0[:, None, None] + (s1 - s0)[:, None, None] * (x[None, :, None] + 1) / 2
    P = p0[:, None, None] + (p1 - p0)[:, None, None] * (x[None, None, :] + 1) / 2
    W = ((s1 - s0) * (p1 - p0))[:, None, None] * (g[None, :, None] * g[None, None, :]) / 4
    S, P, W = (np.broadcast_to(a, (len(s0), order, order)).reshape(len(s0), -1) for a in (S, P, W))
    rho = np.exp(S) * w
    cos_h = 1 / np.sqrt(1 + rho * rho)
    wh = np.stack([rho * cos_h * np.cos(P), cos_h, rho * cos_h * np.sin(P)], -1)
    wo = np.asarray(wo_l, np.float64)
    d = (wh * wo).sum(-1)
    dwh = W * rho * rho * cos_h ** 3
    return 2 * d[..., None] * wh - wo, dwh * 4 * np.abs(d), wh, dwh
