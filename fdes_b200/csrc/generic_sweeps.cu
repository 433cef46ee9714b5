// fdes_b200 -- the multislice sweeps for ANY grid size, even or odd (run-time N): the fallback behind the
// register-resident kernels of sweep_kernels.cuh, which exist for a fixed list of sizes
// (sweep_vtable.h).  The reference accepts every sample size m = n + 2 dn (src/paramStructure.cu:650-651,
// cufftPlan2d at :676-679), e.g. image_size 600 or 675 + 2 * 100; those grids run here.
//
// Same sweeps, same data layout, same tables and scale conventions as the fast path (so the engine does
// not know which one it drives); what differs is the line transform: a mixed-radix Stockham FFT
// in shared memory whose radices are the prime factors of N (pairs of 2 merged to 4), every butterfly
// evaluated as a direct DFT with twiddles from one table W[k] = exp(-2 pi i k / N) computed in double
// precision.  O(N sum r_i) per line instead of O(N log N), which is irrelevant next to correctness for
// a fallback, and it needs no per-size code.  A CTA owns one row, or L = 4 / 2 / 1 adjacent columns.
// The 2/3 band limit is applied by the mask only: no column is skipped (SweepGeom::lo_end = hi_start = N).
#include "sweep_vtable.h"
#include <algorithm>
#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

namespace fdes {
namespace {

constexpr int GT = 256;          // threads per CTA
constexpr int MAXFAC = 24;
struct GPlan {
    int N, nfac;
    int fac[MAXFAC];
};

GPlan make_plan(int N)
{
    GPlan p{};
    p.N = N;
    int n = N, twos = 0;
    while (n % 2 == 0) { twos++; n /= 2; }
    for (; twos >= 2; twos -= 2) p.fac[p.nfac++] = 4;
    if (twos) p.fac[p.nfac++] = 2;
    for (int d = 3; (long long)d * d <= n; d += 2)
        while (n % d == 0) { p.fac[p.nfac++] = d; n /= d; }
    if (n > 1) p.fac[p.nfac++] = n;
    if (p.nfac == 0) p.fac[p.nfac++] = 1;
    return p;
}

__device__ __forceinline__ cpx cmulg(cpx a, cpx b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ int iwg(int i, int N) { return i > N / 2 ? i - N : i; }

// L lines of N points each, a[l * N + i]; all threads of the CTA call it; on return `a` holds the
// transform (the two buffers are swapped as needed).  dir = -1 forward, +1 unnormalised inverse.
__device__ void g_fft(cpx*& a, cpx*& b, const GPlan& pl, int L, const cpx* __restrict__ W, int dir)
{
    const int N = pl.N;
    int Ns = 1;
    for (int f = 0; f < pl.nfac; f++) {
        const int r = pl.fac[f];
        if (r == 1) break;
        const int M = N / r;                 // butterflies per line
        const int step = N / (Ns * r);       // twiddle exponent unit of this pass
        const int dstep = N / r;             // exponent unit of the radix-r DFT matrix
        // Wd: the same table in double precision (appended to W, see gen_twiddles).  Long direct DFTs (prime
        // factors beyond 16, e.g. N = 499) multiply and accumulate in double: a float32 sum of hundreds of
        // terms loses a digit that the O(log N) stages of cuFFT keep.
        const double* Wd = reinterpret_cast<const double*>(W + N);      // 8-byte aligned for any N
        for (int w = threadIdx.x; w < L * M * r; w += GT) {
            // one OUTPUT element per work item: (line l, butterfly j, output index s)
            const int s = w % r, j = (w / r) % M, l = w / (r * M);
            const int k = j % Ns;
            int q = k * step + s * dstep;    // exponent increment per input t
            q %= N;
            const cpx* in = a + l * N + j;
            cpx res;
            if (r > 16) {
                double ax = in[0].x, ay = in[0].y;
                int e = q;
                for (int t = 1; t < r; t++) {
                    double2 tw = make_double2(Wd[2 * e], Wd[2 * e + 1]);
                    if (dir > 0) tw.y = -tw.y;
                    const double vx = in[t * M].x, vy = in[t * M].y;
                    ax += vx * tw.x - vy * tw.y;
                    ay += vx * tw.y + vy * tw.x;
                    e += q;
                    if (e >= N) e -= N;
                }
                res = make_float2((float)ax, (float)ay);
            } else {
                cpx acc = in[0];
                int e = q;
                for (int t = 1; t < r; t++) {
                    cpx tw = W[e];
                    if (dir > 0) tw.y = -tw.y;
                    acc = make_float2(acc.x + in[t * M].x * tw.x - in[t * M].y * tw.y,
                                      acc.y + in[t * M].x * tw.y + in[t * M].y * tw.x);
                    e += q;
                    if (e >= N) e -= N;
                }
                res = acc;
            }
            b[l * N + (j - k) * r + k + s * Ns] = res;
        }
        __syncthreads();
        cpx* t = a; a = b; b = t;
        Ns *= r;
    }
}

// rows: line = one row, element i at base + i; cols: L adjacent columns, element (i, l) at base + i*N + l
template <bool COLS>
__device__ __forceinline__ size_t gaddr(int i, int l, int N) { return COLS ? (size_t)i * N + l : (size_t)i; }
template <bool COLS, class F>
__device__ __forceinline__ void g_foreach(int N, int L, F f)
{
    // cols: consecutive threads walk the L columns of a row first (coalesced L*8-byte segments)
    for (int w = threadIdx.x; w < L * N; w += GT) {
        const int l = COLS ? w % L : 0, i = COLS ? w / L : w;
        f(i, l);
    }
}
struct Smem3 {
    cpx *a, *b, *c;
    __device__ Smem3(cpx* base, int n) : a(base), b(base + n), c(base + 2 * n) {}
};

// ---- S1 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_density_rows(cpx* A, const int* rowptr, const int* rec_col, const float* rec_w,
                                                     int slice, int slice2, int nZ, size_t rec_stride, size_t rp_stride,
                                                     int cfg_stride, int cfg_off2, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, row = blockIdx.x, z = blockIdx.y, b = blockIdx.z;
    cpx *x = gsm, *y = gsm + N;
    const int bA = b * cfg_stride, bB = bA + cfg_off2;      // configurations of the two parts (sweep_kernels.cuh)
    const int* rp = rowptr + (size_t)bA * rp_stride + (size_t)(slice * nZ + z) * N;
    const int lo = rp[row], hi = rp[row + 1];
    int lo2 = 0, hi2 = 0;
    if (slice2 >= 0) {
        const int* rp2 = rowptr + (size_t)bB * rp_stride + (size_t)(slice2 * nZ + z) * N;
        lo2 = rp2[row]; hi2 = rp2[row + 1];
    }
    if (hi <= lo && hi2 <= lo2) return;       // S2 reads such rows as zero
    for (int i = threadIdx.x; i < N; i += GT) x[i] = make_float2(0.f, 0.f);
    __syncthreads();
    if (threadIdx.x == 0) {                   // sorted order: deterministic sums
        const int* cc = rec_col + (size_t)bA * rec_stride;
        const float* ww = rec_w + (size_t)bA * rec_stride;
        for (int i = lo; i < hi; i++) x[cc[i]].x += ww[i];
        const int* cc2 = rec_col + (size_t)bB * rec_stride;
        const float* ww2 = rec_w + (size_t)bB * rec_stride;
        for (int i = lo2; i < hi2; i++) x[cc2[i]].y += ww2[i];
    }
    __syncthreads();
    g_fft(x, y, pl, 1, W, -1);
    cpx* out = A + ((size_t)(b * nZ + z) * N + row) * N;
    for (int i = threadIdx.x; i < N; i += GT) out[i] = x[i];
}

// ---- S2 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_potential_cols(cpx* B, const cpx* A, const float* Gq, const int* rowptr, int slice,
                                                       int slice2, int nZ, size_t rp_stride, int cfg_stride, int cfg_off2, int L,
                                                       GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, Q = N / 2 + 1, kx0 = blockIdx.x * L, b = blockIdx.y;
    Smem3 s(gsm, L * N);
    cpx *x = s.a, *y = s.b, *acc = s.c;
    g_foreach<true>(N, L, [&](int i, int l) { acc[l * N + i] = make_float2(0.f, 0.f); });
    bool any = false;
    for (int z = 0; z < nZ; z++) {
        const int bA = b * cfg_stride, bB = bA + cfg_off2;
        const int* rp = rowptr + (size_t)bA * rp_stride + (size_t)(slice * nZ + z) * N;
        const int* rp2 = slice2 >= 0 ? rowptr + (size_t)bB * rp_stride + (size_t)(slice2 * nZ + z) * N : rp;
        if (rp[N] == rp[0] && rp2[N] == rp2[0]) continue;
        const cpx* Az = A + (size_t)(b * nZ + z) * N * N + kx0;
        __syncthreads();
        g_foreach<true>(N, L, [&](int i, int l) {
            const bool keep = (rp[i + 1] > rp[i]) | (rp2[i + 1] > rp2[i]);
            x[l * N + i] = keep ? Az[gaddr<true>(i, l, N)] : make_float2(0.f, 0.f);
        });
        __syncthreads();
        g_fft(x, y, pl, L, W, -1);
        const float* G = Gq + (size_t)z * Q * Q;
        g_foreach<true>(N, L, [&](int i, int l) {
            const int kx = kx0 + l, ax = min(kx, N - kx), ay = min(i, N - i);
            const float gz = G[(size_t)ax * Q + ay];
            const cpx v = x[l * N + i];
            acc[l * N + i] = make_float2(acc[l * N + i].x + v.x * gz, acc[l * N + i].y + v.y * gz);
        });
        any = true;
    }
    __syncthreads();
    if (any) {
        cpx* t = acc;      // transform the accumulator (x / y serve as the second buffer)
        g_fft(t, x, pl, L, W, +1);
        acc = t;
    }
    cpx* out = B + (size_t)b * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { out[gaddr<true>(i, l, N)] = acc[l * N + i]; });
}

// potential2Transmission (src/multisliceSimulation.cu:41-52) with V.x = V, V.y = imPot * V
__device__ __forceinline__ cpx g_transmission(float V, float imPot)
{
    float sn, cs;
    sincosf(V, &sn, &cs);
    if (imPot != 0.f) {
        const float e = expf(-(V * imPot));
        return make_float2(e * cs, e * sn);
    }
    return make_float2(cs, sn);
}

// ---- S3 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_transmit_rows(const cpx* Wf, cpx* D, int npair, float imPot, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N;
    Smem3 s(gsm, N);
    cpx *x = s.a, *y = s.b;
    cpx* park = s.c;
    const size_t row = blockIdx.x, in_off = ((size_t)blockIdx.y * N + row) * N;
    for (int i = threadIdx.x; i < N; i += GT) x[i] = Wf[in_off + i];
    __syncthreads();
    g_fft(x, y, pl, 1, W, +1);
    for (int i = threadIdx.x; i < N; i += GT) park[i] = x[i];      // V_a + i V_b
    __syncthreads();
    for (int p = 0; p < npair; p++) {
        for (int i = threadIdx.x; i < N; i += GT) x[i] = g_transmission(p == 0 ? park[i].x : park[i].y, imPot);
        __syncthreads();
        g_fft(x, y, pl, 1, W, -1);
        cpx* out = D + ((size_t)(blockIdx.y * 2 + p) * N + row) * N;
        for (int i = threadIdx.x; i < N; i += GT) out[i] = x[i];
        __syncthreads();
    }
}

// ---- S4 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_bandlimit_cols(cpx* Wf, int npair, int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, kx0 = blockIdx.x * L;
    cpx *x = gsm, *y = gsm + L * N;
    const size_t entry = npair == 0 ? blockIdx.y : (size_t)(blockIdx.y / npair) * 2 + blockIdx.y % npair;
    cpx* tile = Wf + entry * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { x[l * N + i] = tile[gaddr<true>(i, l, N)]; });
    __syncthreads();
    g_fft(x, y, pl, L, W, -1);
    const float mind = (float)N, alpha = 1.f / ((float)(N * N));
    g_foreach<true>(N, L, [&](int i, int l) {
        const int i1 = iwg(kx0 + l, N), i2 = iwg(i, N);
        const bool cut = ((float)(i1 * i1 + i2 * i2) * 9.f / (mind * mind)) > 1.f;
        const cpx v = x[l * N + i];
        x[l * N + i] = cut ? make_float2(0.f, 0.f) : make_float2(v.x * alpha, v.y * alpha);
    });
    __syncthreads();
    g_fft(x, y, pl, L, W, +1);
    g_foreach<true>(N, L, [&](int i, int l) { tile[gaddr<true>(i, l, N)] = x[l * N + i]; });
}

// ---- S5 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_multiply_rows(cpx* Psi, const cpx* Tk, size_t e_batch_stride, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N;
    Smem3 s(gsm, N);
    cpx *x = s.a, *y = s.b;
    cpx* park = s.c;
    const size_t row = blockIdx.x;
    const cpx* e = Tk + (size_t)blockIdx.y * e_batch_stride + row * N;
    cpx* p = Psi + ((size_t)blockIdx.y * N + row) * N;
    for (int i = threadIdx.x; i < N; i += GT) x[i] = e[i];
    __syncthreads();
    g_fft(x, y, pl, 1, W, +1);
    for (int i = threadIdx.x; i < N; i += GT) park[i] = x[i];
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += GT) x[i] = p[i];
    __syncthreads();
    g_fft(x, y, pl, 1, W, +1);
    for (int i = threadIdx.x; i < N; i += GT) x[i] = cmulg(park[i], x[i]);
    __syncthreads();
    g_fft(x, y, pl, 1, W, -1);
    for (int i = threadIdx.x; i < N; i += GT) p[i] = x[i];
}

// ---- S6 -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_propagate_cols(cpx* Psi, const cpx* Pq, int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, Q = N / 2 + 1, kx0 = blockIdx.x * L;
    cpx *x = gsm, *y = gsm + L * N;
    cpx* tile = Psi + (size_t)blockIdx.y * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { x[l * N + i] = tile[gaddr<true>(i, l, N)]; });
    __syncthreads();
    g_fft(x, y, pl, L, W, -1);
    g_foreach<true>(N, L, [&](int i, int l) {
        const int kx = kx0 + l;
        x[l * N + i] = cmulg(x[l * N + i], Pq[(size_t)min(kx, N - kx) * Q + min(i, N - i)]);
    });
    __syncthreads();
    g_fft(x, y, pl, L, W, +1);
    g_foreach<true>(N, L, [&](int i, int l) { tile[gaddr<true>(i, l, N)] = x[l * N + i]; });
}

// ---- generic row sweep ----------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_rows_fft(const void* in_, void* out_, int dir, int epi, RowOpts o, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, yrow = blockIdx.x;
    cpx *x = gsm, *y = gsm + N;
    const size_t rowoff = ((size_t)blockIdx.y * N + yrow) * N;
    for (int i = threadIdx.x; i < N; i += GT)
        x[i] = o.in_is_real ? make_float2(static_cast<const float*>(in_)[rowoff + i], 0.f) : static_cast<const cpx*>(in_)[rowoff + i];
    __syncthreads();
    g_fft(x, y, pl, 1, W, dir);
    for (int xx = threadIdx.x; xx < N; xx += GT) {
        const cpx v = make_float2(x[xx].x * o.scale, x[xx].y * o.scale);
        if (epi == ROW_STORE) static_cast<cpx*>(out_)[rowoff + xx] = v;
        else if (epi == ROW_ACCUM) {
            cpx* q = static_cast<cpx*>(out_) + rowoff + xx;
            const cpx old = *q;
            *q = make_float2(old.x + v.x, old.y + v.y);
        } else if (epi == ROW_INTENS_ACCUM) {
            float* q = static_cast<float*>(out_) + rowoff + xx;
            *q += o.scale * (x[xx].x * x[xx].x + x[xx].y * x[xx].y);
        } else if (epi == ROW_STORE_SHIFT) {
            const int ys = (yrow + N / 2) % N, xs = (xx + N / 2) % N;
            static_cast<cpx*>(out_)[((size_t)blockIdx.y * N + ys) * N + xs] = v;
        } else {
            const int cx = xx - o.dn1, cy = yrow - o.dn2;
            if (cx >= 0 && cx < o.n1 && cy >= 0 && cy < o.n2)
                static_cast<float*>(out_)[((size_t)blockIdx.y * o.n2 + cy) * o.n1 + cx] = v.x;
        }
    }
}

// fixed-order batch sum (see k_rows_fft_sum): out (+)= sum_b epilogue(IFFT_row(in[b]))
__global__ void __launch_bounds__(GT) g_rows_fft_sum(const cpx* in, void* out_, int epi, RowOpts o, int nb, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, yrow = blockIdx.x;
    Smem3 s(gsm, N);
    cpx *x = s.a, *y = s.b;
    cpx* acc = s.c;
    const size_t rowoff = (size_t)yrow * N;
    for (int i = threadIdx.x; i < N; i += GT)
        acc[i] = epi == ROW_ACCUM ? static_cast<const cpx*>(out_)[rowoff + i] : make_float2(static_cast<const float*>(out_)[rowoff + i], 0.f);
    for (int b = 0; b < nb; b++) {
        const cpx* src = in + (size_t)b * N * N + rowoff;
        __syncthreads();
        for (int i = threadIdx.x; i < N; i += GT) x[i] = src[i];
        __syncthreads();
        g_fft(x, y, pl, 1, W, +1);
        for (int i = threadIdx.x; i < N; i += GT) {
            if (epi == ROW_ACCUM) { acc[i].x += x[i].x * o.scale; acc[i].y += x[i].y * o.scale; }
            else acc[i].x += o.scale * (x[i].x * x[i].x + x[i].y * x[i].y);
        }
    }
    for (int i = threadIdx.x; i < N; i += GT) {
        if (epi == ROW_ACCUM) static_cast<cpx*>(out_)[rowoff + i] = acc[i];
        else static_cast<float*>(out_)[rowoff + i] = acc[i].x;
    }
}

// ---- generic column sweep -------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_cols_fft(const cpx* in, void* out_, int dir, int op, const void* table, float scale,
                                                 int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, kx0 = blockIdx.x * L;
    cpx *x = gsm, *y = gsm + L * N;
    const size_t boff = (size_t)blockIdx.y * N * N;
    g_foreach<true>(N, L, [&](int i, int l) { x[l * N + i] = in[boff + kx0 + gaddr<true>(i, l, N)]; });
    __syncthreads();
    if (op == COL_PLAIN) {
        g_fft(x, y, pl, L, W, dir);
        g_foreach<true>(N, L, [&](int i, int l) {
            static_cast<cpx*>(out_)[boff + kx0 + gaddr<true>(i, l, N)] = make_float2(x[l * N + i].x * scale, x[l * N + i].y * scale);
        });
        return;
    }
    g_fft(x, y, pl, L, W, -1);
    if (op == COL_DP_ACCUM) {
        float* out = static_cast<float*>(out_);
        g_foreach<true>(N, L, [&](int i, int l) {
            const int xs = (kx0 + l + N / 2) % N, ys = (i + N / 2) % N;
            const cpx v = x[l * N + i];
            out[boff + (size_t)ys * N + xs] += scale * (v.x * v.x + v.y * v.y);
        });
        return;
    }
    g_foreach<true>(N, L, [&](int i, int l) {
        const size_t idx = (size_t)i * N + kx0 + l;
        const cpx v = x[l * N + i];
        if (op == COL_MUL_CPX_INV) {
            const cpx w = static_cast<const cpx*>(table)[(size_t)(kx0 + l) * N + i];     // stored [kx][ky]
            x[l * N + i] = make_float2(w.x * v.x - w.y * v.y, w.x * v.y + w.y * v.x);
        } else {
            const float w = static_cast<const float*>(table)[idx];
            x[l * N + i] = make_float2(v.x * w, v.y * w);
        }
    });
    __syncthreads();
    g_fft(x, y, pl, L, W, +1);
    g_foreach<true>(N, L, [&](int i, int l) {
        static_cast<cpx*>(out_)[boff + kx0 + gaddr<true>(i, l, N)] = make_float2(x[l * N + i].x * scale, x[l * N + i].y * scale);
    });
}

// ---- STEM -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GT) g_probe_cols(cpx* Psi, const cpx* PSI0, const float* shifts, int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, kx0 = blockIdx.x * L;
    cpx *x = gsm, *y = gsm + L * N;
    const float sx = shifts[2 * blockIdx.y], sy = shifts[2 * blockIdx.y + 1], inv = 1.f / (float)N;
    g_foreach<true>(N, L, [&](int i, int l) {
        const float a = (float)iwg(kx0 + l, N), b = (float)iwg(i, N);
        float t = fmaf(a, sx, -rintf(a * sx)) + fmaf(b, sy, -rintf(b * sy));   // phase in turns (see k_probe_cols)
        t -= rintf(t);
        float sn, cs;
        sincosf(-6.283185307179586f * t, &sn, &cs);
        x[l * N + i] = cmulg(PSI0[kx0 + gaddr<true>(i, l, N)], make_float2(cs * inv, sn * inv));
    });
    __syncthreads();
    g_fft(x, y, pl, L, W, +1);
    cpx* out = Psi + (size_t)blockIdx.y * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { out[gaddr<true>(i, l, N)] = x[l * N + i]; });
}

__global__ void __launch_bounds__(GT) g_detector_cols(const cpx* Psi, float* partial, DetectorRings rings, float inv_l1, float inv_l2,
                                                      int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, kx0 = blockIdx.x * L;
    cpx *x = gsm, *y = gsm + L * N;
    const cpx* tile = Psi + (size_t)blockIdx.y * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { x[l * N + i] = tile[gaddr<true>(i, l, N)]; });
    __syncthreads();
    g_fft(x, y, pl, L, W, -1);
    float acc[MAX_DETECTORS];
    for (int d = 0; d < MAX_DETECTORS; d++) acc[d] = 0.f;
    g_foreach<true>(N, L, [&](int i, int l) {
        const float k1 = (float)iwg(kx0 + l, N) * inv_l1, k2 = (float)iwg(i, N) * inv_l2;
        const float ksq = k1 * k1 + k2 * k2;
        const cpx v = x[l * N + i];
        const float p = v.x * v.x + v.y * v.y;
        for (int d = 0; d < rings.n; d++)
            if (ksq >= rings.in2[d] && ksq < rings.out2[d]) acc[d] += p;
    });
    __syncthreads();
    float* red = reinterpret_cast<float*>(gsm);      // deterministic tree over the CTA
    for (int d = 0; d < rings.n; d++) {
        red[threadIdx.x] = acc[d];
        __syncthreads();
        for (int s = GT / 2; s > 0; s >>= 1) {
            if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
            __syncthreads();
        }
        if (threadIdx.x == 0) partial[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * MAX_DETECTORS + d] = red[0];
        __syncthreads();
    }
}
// 4D-STEM (see k_detector4d_cols): the window pixels of the L columns, stored from the line buffers row by row
__global__ void __launch_bounds__(GT) g_detector4d_cols(const cpx* Psi, float* scratch, int Q, int L, GPlan pl, const cpx* W)
{
    extern __shared__ cpx gsm[];
    const int N = pl.N, kx0 = blockIdx.x * L, o = (N - Q) / 2;
    bool any = false;
    for (int l = 0; l < L; l++) any |= (unsigned)((kx0 + l + N / 2) % N - o) < (unsigned)Q;
    if (!any) return;                              // CTA-uniform
    cpx *x = gsm, *y = gsm + L * N;
    const cpx* tile = Psi + (size_t)blockIdx.y * N * N + kx0;
    g_foreach<true>(N, L, [&](int i, int l) { x[l * N + i] = tile[gaddr<true>(i, l, N)]; });
    __syncthreads();
    g_fft(x, y, pl, L, W, -1);
    float* out = scratch + (size_t)blockIdx.y * Q * Q;
    g_foreach<true>(N, L, [&](int i, int l) {
        const int qx = (kx0 + l + N / 2) % N - o, qy = (i + N / 2) % N - o;
        const cpx v = x[l * N + i];
        if ((unsigned)qx < (unsigned)Q && (unsigned)qy < (unsigned)Q) out[(size_t)qy * Q + qx] = v.x * v.x + v.y * v.y;
    });
}
__global__ void g_detector_finish(const float* partial, float* out, int ntiles, int ndet, int batch, float weight)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch * ndet) return;
    const int b = i / ndet, d = i % ndet;
    float s = 0.f;
    for (int t = 0; t < ntiles; t++) s += partial[((size_t)b * ntiles + t) * MAX_DETECTORS + d];
    out[(size_t)b * ndet + d] += weight * s;
}

// ---- host side --------------------------------------------------------------------------------------
size_t smem_limit()
{
    int dev = 0, lim = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    return (size_t)lim;
}
// columns per CTA: the widest of 4, 2, 1 that divides N and fits `bufs` line buffers
int col_width(int N, int bufs)
{
    for (int L : {4, 2, 1})
        if (N % L == 0 && (size_t)L * bufs * N * sizeof(cpx) <= smem_limit()) return L;
    throw std::runtime_error("grid size " + std::to_string(N) + " too large for the generic sweeps");
}
void check_geom(const SweepGeom& g)
{
    if (g.lo_end < g.N || g.hi_start < g.N)
        throw std::runtime_error("generic sweeps expect the whole column range (lo_end = hi_start = N)");
}
void gen_density_rows(const SweepGeom& g, cpx* A, const int* rowptr, const int* rec_col, const float* rec_w, int slice, int slice2,
                  int nZ, int batch, size_t rec_stride, size_t rp_stride, int cfg_stride, int cfg_off2, cudaStream_t st)
{
    const size_t sm = 2 * (size_t)g.N * sizeof(cpx);
    launch(g_density_rows, dim3(g.N, nZ, batch), GT, sm, st, A, rowptr, rec_col, rec_w, slice, slice2, nZ, rec_stride, rp_stride,
           cfg_stride, cfg_off2, make_plan(g.N), g.tw);
}
void gen_potential_cols(const SweepGeom& g, cpx* B, const cpx* A, const float* Gq, const int* rowptr, int slice, int slice2, int nZ,
                    int batch, size_t rp_stride, int cfg_stride, int cfg_off2, cudaStream_t st)
{
    const int L = col_width(g.N, 3);
    const size_t sm = 3 * (size_t)L * g.N * sizeof(cpx);
    launch(g_potential_cols, dim3(g.N / L, batch), GT, sm, st, B, A, Gq, rowptr, slice, slice2, nZ, rp_stride, cfg_stride, cfg_off2, L,
           make_plan(g.N), g.tw);
}
void gen_transmit_rows(const SweepGeom& g, const cpx* Wf, cpx* D, int npair, float imPot, int batch, cudaStream_t st)
{
    check_geom(g);
    const size_t sm = 3 * (size_t)g.N * sizeof(cpx);
    launch(g_transmit_rows, dim3(g.N, batch), GT, sm, st, Wf, D, npair, imPot, make_plan(g.N), g.tw);
}
void gen_bandlimit_cols(const SweepGeom& g, cpx* Wf, int batch, int npair, cudaStream_t st)
{
    check_geom(g);
    const int L = col_width(g.N, 2);
    const size_t sm = 2 * (size_t)L * g.N * sizeof(cpx);
    launch(g_bandlimit_cols, dim3(g.N / L, npair == 0 ? batch : batch * npair), GT, sm, st, Wf, npair, L, make_plan(g.N), g.tw);
}
void gen_multiply_rows(const SweepGeom& g, cpx* Psi, const cpx* E, size_t e_batch_stride, int batch, bool, cudaStream_t st)
{
    check_geom(g);
    const size_t sm = 3 * (size_t)g.N * sizeof(cpx);
    launch(g_multiply_rows, dim3(g.N, batch), GT, sm, st, Psi, E, e_batch_stride, make_plan(g.N), g.tw);
}
void gen_propagate_cols(const SweepGeom& g, cpx* Psi, const cpx* Pq, int batch, cudaStream_t st)
{
    check_geom(g);
    const int L = col_width(g.N, 2);
    const size_t sm = 2 * (size_t)L * g.N * sizeof(cpx);
    launch(g_propagate_cols, dim3(g.N / L, batch), GT, sm, st, Psi, Pq, L, make_plan(g.N), g.tw);
}
void gen_rows_fft(const SweepGeom& g, const void* in, void* out, int dir, RowEpilogue epi, const RowOpts& o, int batch, cudaStream_t st)
{
    const size_t sm = 2 * (size_t)g.N * sizeof(cpx);
    launch(g_rows_fft, dim3(g.N, batch), GT, sm, st, in, out, dir, (int)epi, o, make_plan(g.N), g.tw);
}
void gen_rows_fft_sum(const SweepGeom& g, const cpx* in, void* out, int dir, RowEpilogue epi, const RowOpts& o, int nb, cudaStream_t st)
{
    if (dir <= 0 || (epi != ROW_ACCUM && epi != ROW_INTENS_ACCUM))
        throw std::runtime_error("launch_rows_fft_sum supports inverse transforms with ROW_ACCUM / ROW_INTENS_ACCUM");
    const size_t sm = 3 * (size_t)g.N * sizeof(cpx);
    launch(g_rows_fft_sum, dim3(g.N), GT, sm, st, in, out, (int)epi, o, nb, make_plan(g.N), g.tw);
}
void gen_cols_fft(const SweepGeom& g, const cpx* in, void* out, int dir, ColOp op, const void* table, float scale, int batch, cudaStream_t st)
{
    const int L = col_width(g.N, 2);
    const size_t sm = 2 * (size_t)L * g.N * sizeof(cpx);
    launch(g_cols_fft, dim3(g.N / L, batch), GT, sm, st, in, out, dir, (int)op, table, scale, L, make_plan(g.N), g.tw);
}
void gen_probe_cols(const SweepGeom& g, cpx* Psi, const cpx* PSI0, const float* shifts, int batch, cudaStream_t st)
{
    check_geom(g);
    const int L = col_width(g.N, 2);
    const size_t sm = 2 * (size_t)L * g.N * sizeof(cpx);
    launch(g_probe_cols, dim3(g.N / L, batch), GT, sm, st, Psi, PSI0, shifts, L, make_plan(g.N), g.tw);
}
int gen_detector_tiles(const SweepGeom& g) { return g.N / col_width(g.N, 2); }
void gen_detector_cols(const SweepGeom& g, const cpx* Psi, float* partial, float* out, const DetectorRings& rings, float d1, float d2,
                   float weight, int batch, cudaStream_t st)
{
    check_geom(g);
    const int L = col_width(g.N, 2), tiles = g.N / L;
    const size_t sm = std::max<size_t>(2 * (size_t)L * g.N * sizeof(cpx), GT * sizeof(float));
    launch(g_detector_cols, dim3(tiles, batch), GT, sm, st, Psi, partial, rings, 1.f / ((float)g.N * d1), 1.f / ((float)g.N * d2), L,
           make_plan(g.N), g.tw);
    const int n = batch * rings.n;
    launch(g_detector_finish, (n + 127) / 128, 128, 0, st, partial, out, tiles, rings.n, batch, weight);
}
void gen_detector4d_cols(const SweepGeom& g, const cpx* Psi, float* scratch, float* out, int Q, int bin, float weight, int batch,
                         cudaStream_t st)
{
    check_geom(g);
    const int L = col_width(g.N, 2);
    const size_t sm = 2 * (size_t)L * g.N * sizeof(cpx);
    launch(g_detector4d_cols, dim3(g.N / L, batch), GT, sm, st, Psi, scratch, Q, L, make_plan(g.N), g.tw);
    launch_detector4d_finish(scratch, out, Q, bin, weight, batch, st);
}
// W[k] = exp(-2 pi i k / N), exact on the axes: N float32 pairs, followed by the same N values as double
// pairs (2 cpx slots each) for the long direct DFTs of g_fft
std::vector<cpx> gen_twiddles(int N)
{
    std::vector<cpx> w((size_t)3 * N);
    double* wd = reinterpret_cast<double*>(w.data() + N);
    for (int k = 0; k < N; k++) {
        double c, s;
        if (k == 0) { c = 1; s = 0; }
        else if (4 * k == N) { c = 0; s = -1; }
        else if (2 * k == N) { c = -1; s = 0; }
        else if (4 * k == 3 * N) { c = 0; s = 1; }
        else {
            const double a = -2.0 * 3.14159265358979323846 * (double)k / (double)N;
            c = cos(a); s = sin(a);
        }
        w[k] = make_float2((float)c, (float)s);
        wd[2 * k] = c; wd[2 * k + 1] = s;
    }
    return w;
}

}  // namespace

// odd sizes too: the half-index convention i > N/2 -> i - N and the quarter tables (index min(k, N - k)
// <= N/2) hold for either parity; a prime N is one direct O(N^2) DFT per line
bool generic_size_supported(int N) { return N >= 8 && N <= 8192; }

const SweepVTable* generic_sweep_vtable()
{
    static const SweepVTable vt = {0, 1, 1, 0, &gen_density_rows, &gen_potential_cols, &gen_transmit_rows, &gen_bandlimit_cols, &gen_multiply_rows,
                                   &gen_propagate_cols, &gen_rows_fft, &gen_rows_fft_sum, &gen_cols_fft, &gen_probe_cols, &gen_detector_tiles,
                                   &gen_detector_cols, &gen_detector4d_cols, &gen_twiddles, nullptr, false};
    return &vt;
}

}  // namespace fdes
