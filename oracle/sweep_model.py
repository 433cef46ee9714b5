"""float64 models of the per-slice sweeps of fdes_b200 (S1..S6 and the sweeps of the image formation
and of the STEM scan).

Written from the sweep contracts (DESIGN.md section 2, the launcher comments of
fdes_b200/csrc/kernels.cuh), not from the kernels:

* grids are [y][x] row-major; between the sweeps a field lives in the mixed (kx, y) domain: array
  index [y][kx].  Row transforms act along the last axis, column transforms along the first;
* transforms are unnormalised: FFT = sum f exp(-2 pi i k n / N), IFFT = sum F exp(+2 pi i k n / N);
* a quarter table (scattering factor Gq, propagator Pq) has (N/2+1)^2 entries tab[|kx|][|ky|] with
  |k| = min(k, N - k) and ky fastest; the CTF table of the image formation is the full [kx][ky] grid;
* columns outside the band [lo_end, hi_start) are never read by the band-limited sweeps (taken as 0)
  and never written by them.  Where a model returns a whole image, the caller compares the band
  columns and checks the others separately.

Everything is complex128 / float64; the models take the product's float32 tables as given.
"""
from __future__ import annotations

import os

import numpy as np
import scipy.fft as sfft

_WORKERS = os.cpu_count() or 1


def fft_rows(a):
    return sfft.fft(np.asarray(a, np.complex128), axis=-1, workers=_WORKERS)


def ifft_rows(a):
    return sfft.ifft(np.asarray(a, np.complex128), axis=-1, norm="forward", workers=_WORKERS)


def fft_cols(a):
    return sfft.fft(np.asarray(a, np.complex128), axis=-2, workers=_WORKERS)


def ifft_cols(a):
    return sfft.ifft(np.asarray(a, np.complex128), axis=-2, norm="forward", workers=_WORKERS)


# ---------------------------------------------------------------------------------------------------
# geometry and tables
# ---------------------------------------------------------------------------------------------------
def band_limits(n: int, fast: bool = True):
    """(lo_end, hi_start) of the band columns: kb = largest |kx| the float32 test of zeroHighFreq keeps on
    the axis, bounds rounded outwards to multiples of 32; (n, n) when the two ranges meet or on the
    generic sweeps (fast = False), which transform every column."""
    if not fast:
        return n, n
    mind2 = np.float32(n) * np.float32(n)
    kb = 0
    while kb + 1 <= n // 2 and not (np.float32((kb + 1) * (kb + 1)) * np.float32(9) / mind2 > np.float32(1)):
        kb += 1
    lo, hi = (kb + 1 + 31) // 32 * 32, (n - kb) // 32 * 32
    return (n, n) if lo >= hi else (lo, hi)


def band_columns(n: int, lo_end: int, hi_start: int) -> np.ndarray:
    kx = np.arange(n)
    return (kx < lo_end) | (kx >= hi_start)


def keep_mask(n: int) -> np.ndarray:
    """The 2/3 limit [ky][kx] with the float32 test of zeroHighFreq: (i1^2 + i2^2) * 9 / N^2 > 1 is cut."""
    i = np.arange(n)
    i = np.where(i > n // 2, i - n, i).astype(np.int64)
    s = (i[:, None] ** 2 + i[None, :] ** 2).astype(np.float32)
    return ~(s * np.float32(9) / (np.float32(n) * np.float32(n)) > np.float32(1))


def quarter_to_full(tab_q: np.ndarray, n: int) -> np.ndarray:
    """Quarter table tab[|kx|][|ky|] ((n/2+1)^2 entries, ky fastest) -> full grid [ky][kx]."""
    q = n // 2 + 1
    t = np.asarray(tab_q).reshape(q, q)
    k = np.arange(n)
    a = np.minimum(k, n - k)
    return t[a[None, :], a[:, None]]          # [ky][kx] = t[|kx|][|ky|]


def full_to_quarter(tab: np.ndarray, n: int) -> np.ndarray:
    """The inverse of quarter_to_full for a table with the quarter symmetry, [|kx|][|ky|] flattened."""
    q = n // 2 + 1
    return np.ascontiguousarray(np.asarray(tab)[:q, :q].T).reshape(-1)


# ---------------------------------------------------------------------------------------------------
# S1..S6
# ---------------------------------------------------------------------------------------------------
def _config_pair(b, cfg_stride, cfg_off2):
    a = b * cfg_stride
    return a, a + cfg_off2


def density(rowptr, cols, w, n, nz, z, slice_, conf):
    """Real density [y][x] of species z in slice `slice_` of configuration `conf` from the sorted records:
    key (slice * nZ + z) * N + y covers records rowptr[conf][key] .. rowptr[conf][key + 1]."""
    rp = np.asarray(rowptr[conf], np.int64)
    k0 = (slice_ * nz + z) * n
    d = np.zeros((n, n))
    rows = np.repeat(np.arange(n), rp[k0 + 1:k0 + n + 1] - rp[k0:k0 + n])
    idx = np.arange(rp[k0], rp[k0 + n])          # the records of one key group are contiguous
    np.add.at(d, (rows, cols[conf][idx]), w[conf][idx].astype(np.float64))
    return d


def deposit_rows(rowptr, n, nz, z, slice_, conf):
    """Rows [y] of species z in slice `slice_` of configuration `conf` that hold deposit records."""
    rp = rowptr[conf]
    k0 = (slice_ * nz + z) * n
    return rp[k0 + 1:k0 + n + 1] > rp[k0:k0 + n]


def s1_density_rows(rowptr, cols, w, n, nz, batch, slice_, slice2, cfg_stride=1, cfg_off2=0):
    """S1: A[b][z] = FFT_row(rho(slice of bA) + i rho(slice2 of bB)), bA = b * cfg_stride, bB = bA + cfg_off2.
    Returns (A [batch][nz][N][N], written [batch][nz][N]): rows without deposits in either part may stay
    unwritten (they are exact zeros when written)."""
    A = np.zeros((batch, nz, n, n), np.complex128)
    rows = np.zeros((batch, nz, n), bool)
    for b in range(batch):
        ca, cb = _config_pair(b, cfg_stride, cfg_off2)
        for z in range(nz):
            d = density(rowptr, cols, w, n, nz, z, slice_, ca).astype(np.complex128)
            rows[b, z] = deposit_rows(rowptr, n, nz, z, slice_, ca)
            if slice2 >= 0:
                d = d + 1j * density(rowptr, cols, w, n, nz, z, slice2, cb)
                rows[b, z] |= deposit_rows(rowptr, n, nz, z, slice2, cb)
            A[b, z] = fft_rows(d)
    return A, rows


def s2_potential_cols(A, Gq, rowptr, n, nz, batch, slice_, slice2, cfg_stride=1, cfg_off2=0):
    """S2: B[b] = IFFT_col(sum_z FFT_col(A[b][z]) * G_z), where only the rows with deposit records of either
    slice are read (the others as zero).  A species absent from both slices adds nothing; with no species
    present B[b] is exactly zero."""
    B = np.zeros((batch, n, n), np.complex128)
    G = [quarter_to_full(np.asarray(Gq).reshape(nz, -1)[z], n).astype(np.float64) for z in range(nz)]
    for b in range(batch):
        ca, cb = _config_pair(b, cfg_stride, cfg_off2)
        acc = np.zeros((n, n), np.complex128)
        for z in range(nz):
            keep = deposit_rows(rowptr, n, nz, z, slice_, ca)
            if slice2 >= 0:
                keep = keep | deposit_rows(rowptr, n, nz, z, slice2, cb)
            if not keep.any():
                continue
            a = np.where(keep[:, None], A[b, z], 0)
            acc += fft_cols(a) * G[z]
        B[b] = ifft_cols(acc)
    return B


def transmission(V, imPot):
    """exp(i V (1 + i imPot)) in float64."""
    V = np.asarray(V, np.float64)
    return np.exp(-float(imPot) * V) * np.exp(1j * V)


def s3_transmit_rows(W, npair, imPot):
    """S3: V_a + i V_b = IFFT_row(W[b]); D[2b + p] = FFT_row(exp(i V_p (1 + i imPot))) for p < npair.
    Returns D [2 batch][N][N] (the slots p >= npair are not written; NaN here)."""
    batch, n, _ = W.shape
    V = ifft_rows(W)
    D = np.full((2 * batch, n, n), np.nan, np.complex128)
    for b in range(batch):
        for p in range(npair):
            D[2 * b + p] = fft_rows(transmission(V[b].real if p == 0 else V[b].imag, imPot))
    return D, V


def stack_entries(batch, npair):
    """Images of a [batch][2] stack that S4 works on (npair 1 or 2), or all of a plain [batch] stack (0)."""
    return list(range(batch)) if npair == 0 else [2 * b + p for b in range(batch) for p in range(npair)]


def s4_bandlimit_cols(W, npair, batch):
    """S4 on the entries of stack_entries: IFFT_col(FFT_col(W) * keep / N^2).  Returns the full stack (the
    other entries unchanged)."""
    n = W.shape[-1]
    out = np.array(W, np.complex128)
    m = keep_mask(n) / float(n * n)
    for e in stack_entries(batch, npair):
        out[e] = ifft_cols(fft_cols(W[e]) * m)
    return out


def s5_multiply_rows(Psi, E, e_stride, band, psi_full):
    """S5: t = IFFT_row(E[b * e_stride]), psi = IFFT_row(Psi[b]); Psi[b] <- FFT_row(t * psi).  E is read in
    the band columns only, Psi too unless psi_full."""
    batch = Psi.shape[0]
    out = np.empty(Psi.shape, np.complex128)
    for b in range(batch):
        t = ifft_rows(np.where(band, E[b * e_stride], 0))
        p = ifft_rows(Psi[b] if psi_full else np.where(band, Psi[b], 0))
        out[b] = fft_rows(t * p)
    return out


def s6_propagate_cols(Psi, Pq, band, scale=1.0, lens=None):
    """S6: Psi[b] <- IFFT_col(FFT_col(scale * Psi[b]) * P [* lens]), band columns read and written; P from
    the quarter table, lens a full table stored [kx][ky]."""
    n = Psi.shape[-1]
    P = quarter_to_full(Pq, n).astype(np.complex128)
    if lens is not None:
        P = P * np.asarray(lens).reshape(n, n).T
    out = np.empty(Psi.shape, np.complex128)
    for b in range(Psi.shape[0]):
        out[b] = ifft_cols(fft_cols(scale * np.where(band, Psi[b], 0)) * P)
    return out


def s6_propagate_cols_from(src, src_img_stride, batch, Pq, band, times_n, lens=None):
    """out[b] = IFFT_col(FFT_col(c * src[b * src_img_stride]) * P [* lens]), c = N when times_n."""
    n = src.shape[-1]
    sel = np.stack([src[b * src_img_stride] for b in range(batch)])
    return s6_propagate_cols(sel, Pq, band, float(n) if times_n else 1.0, lens)


def cols_mul_cpx_inv(x, table, scale, band):
    """COL_MUL_CPX_INV: out = scale * IFFT_col(FFT_col(in) * tab[kx][ky]); `in` is zero outside the band."""
    n = x.shape[-1]
    T = np.asarray(table).reshape(n, n).T
    return np.stack([scale * ifft_cols(fft_cols(np.where(band, xb, 0)) * T) for xb in x])


def cols_dp_accum(x, out, scale):
    """COL_DP_ACCUM: out[b][(ky + N/2) % N][(kx + N/2) % N] += scale * |FFT_col(in[b])|^2."""
    n = x.shape[-1]
    res = np.array(out, np.float64)
    for b in range(x.shape[0]):
        p = np.abs(fft_cols(x[b])) ** 2
        res[b] += scale * np.roll(p, (n // 2, n // 2), axis=(0, 1))
    return res


def rows_fft_sum(x, out, scale, epi_intensity, band):
    """launch_rows_fft_sum, inverse: out += sum_b scale * IFFT_row(in[b]) (ROW_ACCUM) or
    scale * |IFFT_row(in[b])|^2 (ROW_INTENS_ACCUM), band columns of `in` only when band is not None."""
    res = np.array(out, np.complex128 if not epi_intensity else np.float64)
    for xb in x:
        v = ifft_rows(xb if band is None else np.where(band, xb, 0))
        res += scale * (np.abs(v) ** 2 if epi_intensity else v)
    return res


def plane_wave_rowspace(n, batch=1):
    """psi = 1 in the (kx, y) domain, Psi = FFT_row(psi) / N: 1 in column 0."""
    P = np.zeros((batch, n, n), np.complex128)
    P[:, :, 0] = 1
    return P


# ---------------------------------------------------------------------------------------------------
# image formation and STEM: generic row / column sweeps, shifted probes, annular detectors
# ---------------------------------------------------------------------------------------------------
ROW_STORE, ROW_ACCUM, ROW_INTENS_ACCUM, ROW_STORE_SHIFT, ROW_CROP_REAL = range(5)


def signed_index(n: int) -> np.ndarray:
    """iw(k): the frequency of index k, k - N for k > N/2."""
    k = np.arange(n)
    return np.where(k > n // 2, k - n, k)


def rows_fft(x, dir, epi, scale, out=None, band_in=None, band_out=None, crop=None):
    """launch_rows_fft: v = scale * FFT_row(x) (dir -1) or scale * IFFT_row(x) (dir +1) per image, then
    ROW_STORE v (0 outside band_out when given), ROW_ACCUM out + v, ROW_INTENS_ACCUM out + scale * |FFT(x)|^2,
    ROW_STORE_SHIFT v at [(y + N/2) % N][(x + N/2) % N] (numpy's fftshift for either parity), ROW_CROP_REAL
    Re v in the window crop = (dn1, dn2, n1, n2): [dn2:dn2 + n2, dn1:dn1 + n1].  x may be real (in_is_real);
    band_in: only these columns of x are read (the others as zero)."""
    x = np.asarray(x)
    if band_in is not None:
        x = np.where(band_in, x, 0)
    f = fft_rows(x) if dir < 0 else ifft_rows(x)
    v = scale * f
    n = x.shape[-1]
    if epi == ROW_STORE:
        return v if band_out is None else np.where(band_out, v, 0)
    if epi == ROW_ACCUM:
        return np.asarray(out, np.complex128) + v
    if epi == ROW_INTENS_ACCUM:
        return np.asarray(out, np.float64) + scale * np.abs(f) ** 2
    if epi == ROW_STORE_SHIFT:
        return np.roll(v, (n // 2, n // 2), axis=(-2, -1))
    dn1, dn2, n1, n2 = crop
    return v.real[..., dn2:dn2 + n2, dn1:dn1 + n1]


def cols_plain(x, dir, scale):
    """COL_PLAIN: out = scale * FFT_col(x) (dir -1) or scale * IFFT_col(x) (dir +1), every column."""
    return scale * (fft_cols(x) if dir < 0 else ifft_cols(x))


def cols_mul_real_inv(x, table, scale):
    """COL_MUL_REAL_INV: out = scale * IFFT_col(FFT_col(x) * tab[ky][kx]), every column."""
    n = np.asarray(x).shape[-1]
    return scale * ifft_cols(fft_cols(x) * np.asarray(table, np.float64).reshape(n, n))


def probe_phase(n, sx, sy):
    """exp(-2 pi i (iw(kx) sx + iw(ky) sy)) [ky][kx] in float64 for the float32 shift (sx, sy)."""
    w = signed_index(n).astype(np.float64)
    return np.exp(-2j * np.pi * (w[None, :] * float(sx) + w[:, None] * float(sy)))


def probe_cols(PSI0, shifts, band):
    """launch_probe_cols: Psi_b = (1/N) IFFT_col[PSI0 * exp(-2 pi i (iw(kx) sx_b + iw(ky) sy_b))] on the band
    columns (PSI0 [ky][kx] read there only), shifts [batch][2] = (sx, sy) in units of the grid period."""
    P = np.where(band, np.asarray(PSI0).reshape(np.asarray(PSI0).shape[-2:]), 0)
    n = P.shape[-1]
    return np.stack([ifft_cols(P * probe_phase(n, sx, sy)) / n for sx, sy in np.asarray(shifts).reshape(-1, 2)])


def inv_length(n, d):
    """fl32(1 / fl32(N d)): the reciprocal box length the detector launcher computes in float32."""
    return np.float32(1) / (np.float32(n) * np.float32(d))


def detector_ksq(n, inv_l1, inv_l2):
    """|k|^2 [ky][kx] = (iw(kx) inv_l1)^2 + (iw(ky) inv_l2)^2 in float64."""
    w = signed_index(n).astype(np.float64)
    return (w[None, :] * float(inv_l1)) ** 2 + (w[:, None] * float(inv_l2)) ** 2


def detector_cols(Psi, band, in2, out2, inv_l1, inv_l2, weight, out0):
    """launch_detector_cols: out[b][d] = out0[b][d] + weight * sum |FFT_col(Psi_b)|^2 over the band columns and
    every ky with in2[d] <= |k|^2 < out2[d]."""
    Psi = np.asarray(Psi)
    ksq = detector_ksq(Psi.shape[-1], inv_l1, inv_l2)
    inten = np.abs(fft_cols(np.where(band, Psi, 0))) ** 2
    res = np.array(out0, np.float64)
    for d, (a, b) in enumerate(zip(in2, out2)):
        m = band[None, :] & (ksq >= float(a)) & (ksq < float(b))
        res[:, d] += float(weight) * (inten * m).sum(axis=(-2, -1))
    return res
