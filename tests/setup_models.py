"""Float64 models of the set-up, per-pixel and atom kernels (setup_kernels.cu, atoms.cu) and the float32
restatements of the oracle they are compared with.  Inputs are float32 values taken exactly; every model evaluates
the formula in float64, so its distance to the kernel is the kernel's own rounding.

Index conventions follow the kernels: quarter tables [|kx|][|ky|] (ky fastest), full tables [ky][kx] with the
signed frequency index (i > N/2 -> i - N), real-space images [y][x]."""
import numpy as np

import fdes_oracle as orc

f32 = np.float32
EPS32 = float(np.finfo(np.float32).eps)
PI32 = float(f32(3.1415927))          # the engine's pi (Params::cst_pi)
FLT_EPS = float(orc.FLT_EPSILON)


def iw(n):
    i = np.arange(n)
    return np.where(i > n // 2, i - n, i).astype(np.float64)


def params(n, d1, d2, **kw):
    """oracle Params of an n x n grid with pixel sizes d1, d2 (float32) and any other field set."""
    p = orc.Params()
    p.m1 = p.m2 = n
    p.d1, p.d2 = f32(d1), f32(d2)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


# ---- quarter tables --------------------------------------------------------------------------------------
def kirkland64(Z):
    """(a, b, c, d) of oracle/kirkland_table.txt (the fallback outside 1..103) as float64 of the float32 values."""
    return tuple(np.asarray(v, np.float64) for v in orc.kirkland_params(Z))


def scatter_q64(Z, n, d1, d2, sigma):
    """Gq[|kx|][|ky|]: Kirkland f(q) * 4.78776452e-9 sigma / (d1 d2 N^2) [A] / (sinc sinc), float64."""
    a, b, c, d = kirkland64(Z)
    i = np.arange(n // 2 + 1, dtype=np.float64)
    d1a, d2a = 1e10 * float(f32(d1)), 1e10 * float(f32(d2))
    q1 = (i / (d1a * n))[:, None]
    q2 = (i / (d2a * n))[None, :]
    qsq = q1 * q1 + q2 * q2
    f = sum(a[k] / (qsq + b[k]) + c[k] * np.exp(-d[k] * qsq) for k in range(3))
    V = f * (float(f32(4.78776452e-9)) * float(f32(sigma))) / (d1a * d2a * n * n)
    u = PI32 * i / n
    s = (u + FLT_EPS) / (np.sin(u) + FLT_EPS)
    return (V * s[:, None] * s[None, :]).reshape(-1)


def scatter_q32(Z, n, d1, d2, sigma):
    """The non-negative quadrant of the oracle's float32 scattering_factor, as a quarter table."""
    full = orc.scattering_factor(Z, params(n, d1, d2, sigma=f32(sigma), pi=f32(PI32)))
    q = n // 2 + 1
    return np.ascontiguousarray(full[:q, :q].T).reshape(-1)


def prop_q64(n, d1, d2, d3, lam):
    """Pq[|kx|][|ky|] = exp(-i pi lambda d3 |k|^2) / N^2 (mask not applied) and the phase, float64."""
    i = np.arange(n // 2 + 1, dtype=np.float64)
    d1, d2, d3, lam = (float(f32(v)) for v in (d1, d2, d3, lam))
    t1 = (i / n * (d3 / d1))[:, None]
    t2 = (i / n * (d3 / d2))[None, :]
    ph = -PI32 * (t1 * t1 + t2 * t2) * (lam / d3)
    return (np.exp(1j * ph) / (n * n)).reshape(-1), ph.reshape(-1)


def prop_mask_q(n):
    """zeroHighFreq's float32 test on the quarter: keep unless (float)(i1^2 + i2^2) * 9 / N^2 > 1."""
    i = np.arange(n // 2 + 1, dtype=np.int64)
    s = (i[:, None] ** 2 + i[None, :] ** 2).astype(np.float32)
    return ~((s * f32(9)) / (f32(n) * f32(n)) > f32(1)).reshape(-1)


def prop_mask_exact_q(n):
    i = np.arange(n // 2 + 1, dtype=np.int64)
    return ~(9 * (i[:, None] ** 2 + i[None, :] ** 2) > n * n).reshape(-1)


def prop_q32(n, d1, d2, d3, lam):
    p = params(n, d1, d2, d3=f32(d3), lam=f32(lam), pi=f32(PI32))
    full = orc.fresnel_propagator(p)
    q = n // 2 + 1
    return np.ascontiguousarray(full[:q, :q].T).reshape(-1)


# ---- lens table ------------------------------------------------------------------------------------------
def lens_nu(n, d1, d2, lam):
    """(nu1, nu2) [ky][kx] in float64 with the row index pointing up (i2 -> -i2)."""
    nu1 = (iw(n) / n * (float(f32(lam)) / float(f32(d1))))[None, :]
    nu2 = (-iw(n) / n * (float(f32(lam)) / float(f32(d2))))[:, None]
    return np.broadcast_arrays(nu1, nu2)


def lens_nu32_candidates(n, d1, d2, lam):
    """|nu| as the kernel may round it: nu1, nu2 in float32, then sqrtf of nu1^2 + nu2^2 with no contraction or with
    either product fused into the add.  Returns the three candidates [ky][kx]."""
    lamf = f32(lam)
    i = iw(n).astype(np.float32)
    nu1 = ((i / f32(n)).astype(f32) * f32(lamf / f32(d1))).astype(f32)[None, :]
    nu2 = ((-i / f32(n)).astype(f32) * f32(lamf / f32(d2))).astype(f32)[:, None]
    nu1, nu2 = np.broadcast_arrays(nu1, nu2)
    a, b = nu1.astype(np.float64) ** 2, nu2.astype(np.float64) ** 2       # exact
    plain = (nu1 * nu1).astype(f32) + (nu2 * nu2).astype(f32)
    fa = (a + (nu2 * nu2).astype(f32)).astype(f32)
    fb = (b + (nu1 * nu1).astype(f32)).astype(f32)
    return [np.sqrt(v.astype(f32)).astype(f32) for v in (plain, fa, fb)]


def lens64(n, ab0, ab1, defocus, spread, lam, d1, d2, objap, scale, mode):
    """multiplyLensFunction [ky][kx] without the aperture, float64, and the magnitude of chi's terms (the error
    scale).  ab0 / ab1: 14 float32 values."""
    nu1, nu2 = lens_nu(n, d1, d2, lam)
    phi = np.arctan2(nu2, nu1)
    nu = np.hypot(nu1, nu2)
    a0 = [float(f32(v)) for v in ab0]
    a1 = [float(f32(v)) for v in ab1]

    def cs(m, k):
        return a0[k] * np.cos(m * (phi - a1[k]))
    t5 = (cs(6, 11) + cs(4, 12) + cs(2, 13) + a0[10]) / 6
    t4 = (cs(5, 7) + cs(1, 8) + cs(3, 9)) / 5 + nu * t5
    t3 = (cs(4, 5) + cs(2, 6) + a0[4]) / 4 + nu * t4
    t2 = (cs(3, 2) + cs(1, 3)) / 3 + nu * t3
    t1 = (cs(2, 1) + a0[0] + float(f32(defocus))) / 2 + nu * t2
    W = nu * nu * t1
    lam = float(f32(lam))
    env = np.exp(-2 * (float(f32(spread)) * nu * nu / lam) ** 2) if mode == 0 else np.ones_like(nu)
    chi = 2 * PI32 * W / lam
    # the size of chi's terms before they cancel (every cosine at 1, every term positive, times its order for the
    # error of phi): the scale of the rounding error of any evaluation of W
    A = [abs(v) for v in a0]
    Wmag = nu * nu * ((2 * A[1] + A[0] + abs(float(f32(defocus)))) / 2
                      + nu * ((3 * A[2] + A[3]) / 3 + nu * ((4 * A[5] + 2 * A[6] + A[4]) / 4
                      + nu * ((5 * A[7] + A[8] + 3 * A[9]) / 5 + nu * (6 * A[11] + 4 * A[12] + 2 * A[13] + A[10]) / 6))))
    return env * np.exp(-1j * chi) * float(f32(scale)), 2 * PI32 * Wmag / lam


# ---- detector table --------------------------------------------------------------------------------------
def detector64(n, mtf4, illangle, defocus, lam, d1, d2, scale, mode, use_inc, use_mtf):
    """[ky][kx] spatial incoherence (optional) * MTF (optional) * scale and the largest exponent, float64."""
    mtfa, mtfb, mtfc, mtfd = (float(f32(v)) for v in mtf4)
    lam, d1, d2, ill, df = (float(f32(v)) for v in (lam, d1, d2, illangle, defocus))
    i1, i2 = iw(n)[None, :], iw(n)[:, None]
    arg = np.zeros((n, n))
    f = np.ones((n, n))
    if use_inc:
        if mode == 0:
            arg = ((i1 / n * lam / d1) ** 2 + (i2 / n * lam / d2) ** 2) * (PI32 * ill * df) ** 2
        else:
            arg = ((i1 * d1) ** 2 + (i2 * d2) ** 2) * (PI32 * ill / lam) ** 2
        f = np.exp(-arg)
    if use_mtf:
        nu1, nu2 = i1 / n, i2 / n
        r = np.sqrt(nu1 ** 2 + nu2 ** 2)
        m = mtfa * np.exp(-mtfc * r) + mtfb * np.exp(-mtfd * r * r)
        a1, a2 = PI32 * nu1, PI32 * nu2
        m = m * ((np.sin(a1) + FLT_EPS) / (a1 + FLT_EPS)) * ((np.sin(a2) + FLT_EPS) / (a2 + FLT_EPS))
        f = f * m
        arg = arg + mtfc * r + mtfd * r * r
    return f * float(f32(scale)), arg


def detector32(n, mtf4, illangle, defocus, lam, d1, d2, scale, mode, use_inc, use_mtf):
    p = params(n, d1, d2, mtfa=f32(mtf4[0]), mtfb=f32(mtf4[1]), mtfc=f32(mtf4[2]), mtfd=f32(mtf4[3]),
               illangle=f32(illangle), lam=f32(lam), mode=mode, pi=f32(PI32))
    p.defoci = np.array([defocus], np.float32)
    f = np.ones((n, n), np.float32)
    if use_inc:
        f = orc.spatial_incoherence(p, 0)
    if use_mtf:
        f = (f * orc.mtf(p)).astype(f32)
    return (f * f32(scale)).astype(f32)


# ---- real-space per-pixel kernels ------------------------------------------------------------------------
def tilt_phase64(n, d1, d2, lam, tbx, tby, flag):
    """tiltBeam_d phase [y][x]: 2 pi (i1 d1 tb_y + i2 d2 tb_x) / (lambda flag), i = index - N/2, and the sum of
    the two terms' magnitudes (the scale of the phase's rounding error, the terms may cancel)."""
    i = np.arange(n, dtype=np.float64) - n // 2
    d1, d2, lam, tbx, tby = (float(f32(v)) for v in (d1, d2, lam, tbx, tby))
    a = (i * d1 * tby / (lam * flag))[None, :]
    b = (i * d2 * tbx / (lam * flag))[:, None]
    return 2 * PI32 * (a + b), 2 * PI32 * (np.abs(a) + np.abs(b))


def tilt32(psi, n, d1, d2, lam, tbx, tby, flag):
    p = params(n, d1, d2, lam=f32(lam), pi=f32(PI32))
    p.tiltbeam = np.array([tbx, tby], np.float32)
    return orc.tilt_beam(psi, p, 0, flag)


def tukey1d64(n, dn):
    x = np.arange(n, dtype=np.float64) / (n - 1)
    w = np.ones(n)
    if dn == 0:
        return w
    alpha = 2 * dn / n
    lo = x < alpha / 2
    hi = ~lo & (x > 1 - alpha / 2)
    w[lo] = 0.5 * (1 + np.cos(PI32 * (2 * x[lo] / alpha - 1)))
    w[hi] = 0.5 * (1 + np.cos(PI32 * (2 * x[hi] / alpha + 1 - 2 / alpha)))
    return w


def tukey64(n, dn1, dn2):
    return tukey1d64(n, dn2)[:, None] * tukey1d64(n, dn1)[None, :]


def tukey_err_scale(n, dn1, dn2):
    """The reference's upper taper evaluates 2x/alpha + 1 - 2/alpha, alpha = 2 dn / N: its float32 rounding error
    grows with N / dn."""
    return 1 + sum(n / dn for dn in (dn1, dn2) if dn)


def tukey32(psi, n, dn1, dn2):
    return orc.tapered_cosine_window(psi, params(n, 1e-11, 1e-11, dn1=dn1, dn2=dn2, pi=f32(PI32)))


def area1d64(n, dn):
    i = np.arange(n, dtype=np.float64)
    w = np.ones(n)
    if dn == 0:
        return w
    pi = float(f32(3.1415927))
    w = np.where(i <= dn - 1, w * 0.5 * (1 - np.cos(pi * i / dn)), w)
    w = np.where(i >= n - dn, w * 0.5 * (1 - np.cos(pi * (n - i) / dn)), w)
    return w


def area64(n, dn1, dn2):
    return area1d64(n, dn2)[:, None] * area1d64(n, dn1)[None, :]


def area_blend32(psi, n, dn1, dn2):
    am = orc.area_mask(params(n, 1e-11, 1e-11, dn1=dn1, dn2=dn2))
    return ((f32(1) * (f32(1) - am)).astype(f32) + psi * am).astype(np.complex64)


# ---- random numbers ----------------------------------------------------------------------------------------
def box_muller64(x, y):
    """curand_normal's first value of a pair from two raw XORWOW words, in float64 (the device uses logf and
    __sincosf; this is the exact formula)."""
    u = x.astype(np.float64) * 2.0 ** -32 + 2.0 ** -33
    v = y.astype(np.float64) * (2.0 ** -32 * 2 * np.pi) + 2.0 ** -33 * 2 * np.pi
    s = np.sqrt(-2 * np.log(u))
    return s * np.sin(v), s * np.cos(v)


def anscombe32(fi, nrm, dose):
    """ascombeNoise_d on one lit pixel (fi = f * dose > 1e-2) with the normal nrm, float32; returns (out, arg)
    where arg is the value roundf rounds."""
    fi = np.asarray(fi, f32)
    n = np.asarray(nrm, f32)
    with np.errstate(invalid="ignore", divide="ignore"):
        v = (n * np.sqrt((f32(1) - np.exp((-fi / f32(0.777134)).astype(f32))).astype(f32))).astype(f32)
        v = (v + (f32(2) * np.sqrt((fi + f32(0.375)).astype(f32)) - f32(0.25) / np.sqrt(fi)).astype(f32)).astype(f32)
        arg = (f32(0.25) * v * v - f32(0.375)).astype(f32)
    x = orc.roundf(arg)
    x = np.where(x < orc.FLT_MIN, f32(0), x).astype(f32)
    return (x / f32(dose)).astype(f32), arg, v


# ---- deposit records --------------------------------------------------------------------------------------
def records_model(xyz, zidx, occ, n, m3, nz, d1, d2, d3):
    """Records of one configuration as k_bin_atoms writes them (float32 arithmetic of squareAtoms_d through
    orc.bin_atoms), stably sorted by key: (keys, cols, w) and the row pointers."""
    p = params(n, d1, d2, d3=f32(d3), m3=m3)
    i1, i2, i3, r1, r2, ok = orc.bin_atoms(xyz, p)
    ok = ok & (i3 >= 0) & (i3 < m3)
    nkeys = m3 * nz * n
    nat = len(zidx)
    keys = np.full((nat, 4), nkeys, np.int64)
    cols = np.zeros((nat, 4), np.int32)
    w = np.zeros((nat, 4), np.float32)
    g1 = np.where(r1 < 0, -1, 1)
    g2 = np.where(r2 < 0, -1, 1)
    a1, a2 = np.abs(r1), np.abs(r2)
    one = f32(1)
    oc = np.asarray(occ, f32)
    kb = (i3.astype(np.int64) * nz + zidx) * n
    rows = [i2, i2 + g2, i2 + g2, i2]
    cc = [i1, i1, i1 + g1, i1 + g1]
    ww = [((one - a1) * (one - a2)).astype(f32) * oc, ((one - a1) * a2).astype(f32) * oc,
          (a1 * a2).astype(f32) * oc, (a1 * (one - a2)).astype(f32) * oc]
    for q in range(4):
        keys[ok, q] = kb[ok] + rows[q][ok]
        cols[ok, q] = cc[q][ok]
        w[ok, q] = ww[q][ok].astype(f32)
    keys, cols, w = keys.reshape(-1), cols.reshape(-1), w.reshape(-1)
    o = np.argsort(keys, kind="stable")
    keys, cols, w = keys[o], cols[o], w[o]
    rowptr = np.searchsorted(keys, np.arange(nkeys + 1), side="left").astype(np.int32)
    return keys.astype(np.uint32), cols, w, rowptr, (i1, i2, i3, ok)


def row_masks(rowptr, nkeys, n, e):
    """Mask words of launch_row_masks: word theta of key group kg has bit m set when row theta + m T (T = N / E)
    has records."""
    t = n // e
    has = (rowptr[1:nkeys + 1] > rowptr[:nkeys]).reshape(nkeys // n, n)
    words = np.zeros((nkeys // n, t), np.uint64)
    for m in range(e):
        words |= has[:, m * t:(m + 1) * t].astype(np.uint64) << np.uint64(m)
    return words.astype(np.uint32).reshape(-1)
