// fdes_b200 -- set-up kernels: multiplier tables and small utilities.
// The tables are evaluated with the reference's float32 expressions (same operation order,
// precise expf/sinf/cosf, no fast-math) so that they agree with what the reference recomputes
// every slice; here they are computed once per simulation and kept L2-resident.
#include "kernels.cuh"
#include <algorithm>
#include <cfloat>
#include <cstdio>

namespace fdes {

// ---------------------------------------------------------------------------------------------
// scattering factor * sinc correction (projectedPotential_d, src/projectedPotential.cu:30-73;
// divideBySinc, src/crystalMaker.cu:136-158).  Quarter table over |iw| indices.
// ---------------------------------------------------------------------------------------------
__global__ void k_scattering_table(float* __restrict__ Gq, int N, KirklandRow kr, float d1m,
                                   float d2m, float sigma, float pi)
{
    const int Q = N / 2 + 1;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q * Q) return;
    // stored [|kx|][|ky|] (ky fastest): a column sweep's warp reads consecutive ky of ONE kx
    const int i2 = i % Q, i1 = i / Q;
    const int m1 = N, m2 = N;
    const float d1 = 1e10f * d1m;
    const float d2 = 1e10f * d2m;
    // |q|^2 in 1/A^2, Kirkland's parametrisation f(q) = sum_k a_k / (q^2 + b_k) + c_k exp(-d_k q^2)
    const float q1 = ((float)i1) / (d1 * ((float)m1));
    const float q2 = ((float)i2) / (d2 * ((float)m2));
    const float qsq = q1 * q1 + q2 * q2;
    const float* a = kr.v;  // a_k = v[2k], b_k = v[2k+1], c_k = v[6+2k], d_k = v[7+2k]
    float f = a[0] / (qsq + a[1]) + a[6] * expf(-a[7] * qsq);
    f += a[2] / (qsq + a[3]) + a[8] * expf(-a[9] * qsq);
    f += a[4] / (qsq + a[5]) + a[10] * expf(-a[11] * qsq);
    const float V = f * (4.78776452e-9f * sigma) / (d1 * d2 * ((float)(m1 * m2)));
    // 1 / (sinc sinc) of the bilinear deposit, both arguments guarded by FLT_EPSILON as in divideBySinc
    const float u1 = ((float)i1) / ((float)m1) * pi;
    const float inv_sinc1 = (u1 + FLT_EPSILON) / (sinf(u1) + FLT_EPSILON);
    const float u2 = pi * (((float)i2) / ((float)m2));
    const float inv_sinc = inv_sinc1 * ((u2 + FLT_EPSILON) / (sinf(u2) + FLT_EPSILON));
    Gq[i] = V * inv_sinc;
}

static const KirklandRow kKirkland[103] = {
#include "kirkland_table.inc"
};

KirklandRow kirkland_row(int Z)
{
    if (Z >= 1 && Z <= 103) return kKirkland[Z - 1];
    return KirklandRow{{0, 1, 0, 1, 0, 1, 1, 0, 1, 0, 1, 0}};
}

void launch_scattering_table(float* Gq, int N, KirklandRow kr, float d1, float d2, float sigma,
                             float pi, cudaStream_t st)
{
    const int Q = N / 2 + 1, n = Q * Q;
    launch(k_scattering_table, (n + 255) / 256, 256, 0, st, Gq, N, kr, d1, d2, sigma, pi);
}

// ---------------------------------------------------------------------------------------------
// Fresnel propagator with the 2/3 mask and 1/N (fresnelPropagatorDevice + zeroHighFreq + Csscal,
// src/multisliceSimulation.cu:253-274, 225-250, 594-603).  Quarter table.
// ---------------------------------------------------------------------------------------------
__global__ void k_propagator_table(cpx* __restrict__ Pq, int N, float d1, float d2, float d3in,
                                   float lambda, float pi)
{
    const int Q = N / 2 + 1;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q * Q) return;
    const int i2 = i % Q, i1 = i / Q;    // stored [|kx|][|ky|], ky fastest (see k_scattering_table)
    const int dim1 = N, dim2 = N;
    const float d3 = d3in;
    const float t1 = ((float)(i1) / ((float)dim1)) * (d3 / d1);
    const float t2 = ((float)(i2) / ((float)dim2)) * (d3 / d2);
    const float lambda_over_d3 = lambda / d3;
    const float phase = -pi * (t1 * t1 + t2 * t2) * lambda_over_d3;       // -pi lambda dz |k|^2
    cpx p = make_float2(cosf(phase), sinf(phase));
    const float mindim = (float)N;
    if (((float)(i1 * i1 + i2 * i2) * 9.f / (mindim * mindim)) > 1.f) p = make_float2(0.f, 0.f);
    const float alpha = 1.f / ((float)(N * N));
    Pq[i] = make_float2(p.x * alpha, p.y * alpha);
}

void launch_propagator_table(cpx* Pq, int N, float d1, float d2, float d3, float lambda, float pi,
                             cudaStream_t st)
{
    const int Q = N / 2 + 1, n = Q * Q;
    launch(k_propagator_table, (n + 255) / 256, 256, 0, st, Pq, N, d1, d2, d3, lambda, pi);
}

// ---------------------------------------------------------------------------------------------
// lens function (multiplyLensFunction, src/multisliceSimulation.cu:277-343): full table, the
// factor the wave is multiplied with; zero outside the objective aperture.
// ---------------------------------------------------------------------------------------------
// transposed: the entry of (kx, ky) is stored at kx * N + ky (ky fastest), the order in which the T
// threads of a column sweep read it (COL_MUL_CPX_INV); otherwise at ky * N + kx like an image
__global__ void k_lens_table(cpx* __restrict__ tab, int N, LensParams lp, float extra_scale, int transposed)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * N) return;
    int i1 = transposed ? i / N : i % N, i2 = transposed ? i % N : i / N;
    if (i1 > N / 2) i1 -= N;
    if (i2 > N / 2) i2 -= N;
    i2 = -i2;  // row index points up
    const float dim1 = (float)N, dim2 = (float)N;
    // scattering angle (nu1, nu2) = lambda k, its azimuth phi and magnitude nu
    const float nu1 = (((float)i1) / dim1) * (lp.lambda / lp.d1);
    const float nu2 = (((float)i2) / dim2) * (lp.lambda / lp.d2);
    const float phi = atan2f(nu2, nu1);
    const float nu = sqrtf(nu1 * nu1 + nu2 * nu2);
    cpx out = make_float2(0.f, 0.f);
    if (nu < lp.ObjAp) {
        // index: 0 C1, 1 A1, 2 A2, 3 B2, 4 C3, 5 A3, 6 S3, 7 A4, 8 B4, 9 D4, 10 C5, 11 A5, 12 R5, 13 S5
        const float* a0 = lp.ab0;
        const float* a1 = lp.ab1;
        float W = nu * nu * (0.5f * (a0[1] * cosf(2.f * (phi - a1[1])) + a0[0] + lp.defocus_k)
            + nu * (1.f / 3.f * (a0[2] * cosf(3.f * (phi - a1[2])) + a0[3] * cosf(phi - a1[3]))
            + nu * (0.25f * (a0[5] * cosf(4.f * (phi - a1[5])) + a0[6] * cosf(2.f * (phi - a1[6])) + a0[4])
            + nu * (0.2f * (a0[7] * cosf(5.f * (phi - a1[7])) + a0[8] * cosf(phi - a1[8]) + a0[9] * cosf(3.f * (phi - a1[9])))
            + nu * (1.f / 6.f * (a0[11] * cosf(6.f * (phi - a1[11])) + a0[12] * cosf(4.f * (phi - a1[12]))
                                 + a0[13] * cosf(2.f * (phi - a1[13])) + a0[10]))))));
        // aperture * temporal-coherence envelope * exp(-i chi), chi = 2 pi W / lambda
        float envelope = 1.f;
        if (lp.mode == 0) {
            const float spread = lp.defocspread * nu * nu / lp.lambda;
            envelope = expf(-2.f * spread * spread);
        }
        const float chi_over_2pi = W / lp.lambda;
        const float re = envelope * cosf(2.f * lp.pi * chi_over_2pi);
        const float im = envelope * sinf(-2.f * lp.pi * chi_over_2pi);
        out = make_float2(re * extra_scale, im * extra_scale);
    }
    tab[i] = out;
}

void launch_lens_table(cpx* tab, int N, const LensParams& lp, float extra_scale, cudaStream_t st, bool transposed)
{
    const int n = N * N;
    launch(k_lens_table, (n + 255) / 256, 256, 0, st, tab, N, lp, extra_scale, transposed ? 1 : 0);
}

// ---------------------------------------------------------------------------------------------
// detector table: spatial incoherence (optional) * MTF * scale
// (multiplySpatialIncoherence / ...DP / multiplyMtf, src/multisliceSimulation.cu:362-442)
// ---------------------------------------------------------------------------------------------
__global__ void k_detector_table(float* __restrict__ tab, int N, DetectorParams dp, float scale)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * N) return;
    int i1 = i % N, i2 = i / N;
    if (i1 > N / 2) i1 -= N;
    if (i2 > N / 2) i2 -= N;
    const float dim1 = (float)N, dim2 = (float)N;
    float f = 1.f;
    if (dp.use_incoherence) {
        if (dp.mode == 0) {
            float damp = dp.lambda;
            float nusq = (((float)i1) / dim1) * (damp / dp.d1);
            damp = (((float)i2) / dim2) * (damp / dp.d2);
            nusq = nusq * nusq + damp * damp;
            damp = dp.pi * dp.illangle * dp.defocus_k;
            f = expf(-nusq * damp * damp);
        } else {
            float x1 = ((float)i1) * dp.d1;
            float x2 = ((float)i2) * dp.d2;
            x1 = x1 * x1 + x2 * x2;
            x2 = dp.pi * dp.illangle / dp.lambda;
            f = expf(-x2 * x2 * x1);
        }
    }
    float nu1 = ((float)i1) / dim1;
    float nu2 = ((float)i2) / dim2;
    float mtf = sqrtf(nu1 * nu1 + nu2 * nu2);
    mtf = (dp.mtfa * expf(-dp.mtfc * mtf) + dp.mtfb * expf(-dp.mtfd * mtf * mtf));
    nu1 *= dp.pi;
    nu2 *= dp.pi;
    mtf *= ((sinf(nu1) + FLT_EPSILON) / (nu1 + FLT_EPSILON)) * ((sinf(nu2) + FLT_EPSILON) / (nu2 + FLT_EPSILON));
    tab[i] = dp.use_mtf ? f * mtf * scale : f * scale;
}

void launch_detector_table(float* tab, int N, const DetectorParams& dp, float scale, cudaStream_t st)
{
    const int n = N * N;
    launch(k_detector_table, (n + 255) / 256, 256, 0, st, tab, N, dp, scale);
}

// ---------------------------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------------------------
__global__ void k_fill_cpx(cpx* p, size_t n, cpx v)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = v;
}
__global__ void k_fill_f32(float* p, size_t n, float v)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = v;
}
static int grid_for(size_t n) { size_t g = (n + 255) / 256; return (int)(g > 148 * 8 ? 148 * 8 : (g ? g : 1)); }

void launch_fill_cpx(cpx* p, size_t n, cpx v, cudaStream_t st) { launch(k_fill_cpx, grid_for(n), 256, 0, st, p, n, v); }
void launch_fill_f32(float* p, size_t n, float v, cudaStream_t st) { launch(k_fill_f32, grid_for(n), 256, 0, st, p, n, v); }

// out[b][y][x] += weight * sum of scratch[b][y*bin + r][x*bin + c], r outer, c inner: bins straddle the CTAs of the
// detector sweep, so they are summed here, one thread per output pixel, without atomics
__global__ void k_detector4d_finish(const float* __restrict__ scratch, float* __restrict__ out, int Q, int bin, float weight,
                                    size_t n)
{
    const int S = Q / bin;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % S), y = (int)((i / S) % S);
        const float* src = scratch + (i / ((size_t)S * S)) * Q * Q + (size_t)y * bin * Q + (size_t)x * bin;
        float s = 0.f;
        for (int r = 0; r < bin; r++)
            for (int c = 0; c < bin; c++) s += src[(size_t)r * Q + c];
        out[i] += weight * s;
    }
}
void launch_detector4d_finish(const float* scratch, float* out, int Q, int bin, float weight, int batch, cudaStream_t st)
{
    const size_t n = (size_t)batch * (Q / bin) * (Q / bin);
    launch(k_detector4d_finish, grid_for(n), 256, 0, st, scratch, out, Q, bin, weight, n);
}

__global__ void k_plane_wave_rowspace(cpx* Psi, int N, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        Psi[i] = make_float2((i % N) == 0 ? 1.f : 0.f, 0.f);
}
void launch_plane_wave_rowspace(cpx* Psi, int N, int batch, cudaStream_t st)
{
    const size_t n = (size_t)batch * N * N;
    launch(k_plane_wave_rowspace, grid_for(n), 256, 0, st, Psi, N, n);
}

__global__ void k_scale_cpx(cpx* p, size_t n, float s)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = make_float2(p[i].x * s, p[i].y * s);
}
void launch_scale_cpx(cpx* p, size_t n, float s, cudaStream_t st) { launch(k_scale_cpx, grid_for(n), 256, 0, st, p, n, s); }

__global__ void k_absorptive_factor(cpx* V, size_t n, float imPot)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        V[i] = make_float2(V[i].x, V[i].x * imPot);
}
void launch_absorptive_factor(cpx* V, size_t n, float imPot, cudaStream_t st)
{
    launch(k_absorptive_factor, grid_for(n), 256, 0, st, V, n, imPot);
}

__global__ void k_zero_outband(cpx* Psi, int N, int lo_end, int hi_start, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int kx = (int)(i % N);
        if (kx >= lo_end && kx < hi_start) Psi[i] = make_float2(0.f, 0.f);
    }
}
void launch_zero_outband(cpx* Psi, int N, int lo_end, int hi_start, int batch, cudaStream_t st)
{
    const size_t n = (size_t)batch * N * N;
    launch(k_zero_outband, grid_for(n), 256, 0, st, Psi, N, lo_end, hi_start, n);
}

// deterministic two-stage sum of |p|^2: fixed grid, fixed per-thread strides, tree in shared memory
constexpr int NORM_BLOCKS = 256, NORM_THREADS = 256;
__global__ void k_norm2_stage1(const cpx* __restrict__ p, size_t n, double* __restrict__ partial)
{
    __shared__ double sh[NORM_THREADS];
    double acc = 0.0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const cpx v = p[i];
        acc += (double)v.x * v.x + (double)v.y * v.y;
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = NORM_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
__global__ void k_norm2_stage2(const double* __restrict__ partial, double* __restrict__ result)
{
    __shared__ double sh[NORM_BLOCKS];
    sh[threadIdx.x] = partial[threadIdx.x];
    __syncthreads();
    for (int s = NORM_BLOCKS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) result[0] = sh[0];
}
void launch_norm2(const cpx* p, size_t n, double* partial, double* result, cudaStream_t st)
{
    launch(k_norm2_stage1, NORM_BLOCKS, NORM_THREADS, 0, st, p, n, partial);
    launch(k_norm2_stage2, 1, NORM_BLOCKS, 0, st, partial, result);
}

// tiltBeam_d, src/multisliceSimulation.cu:89-120
__global__ void k_tilt_beam(cpx* psi, int N, float d1, float d2, float lambda, float tb_x,
                            float tb_y, float pi, int flag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * N) return;
    const int i1 = i % N - N / 2, i2 = i / N - N / 2;
    float x2 = lambda * ((float)flag);
    float x1 = ((float)i1) * (d1 / x2) * tb_y;   // tiltbeam[2k+1]
    x2 = ((float)i2) * (d2 / x2) * tb_x;         // tiltbeam[2k]
    x1 = 2.f * pi * (x1 + x2);
    x2 = sinf(x1);
    x1 = cosf(x1);
    const cpx v = psi[i];
    psi[i] = make_float2(x1 * v.x - x2 * v.y, x2 * v.x + x1 * v.y);
}
void launch_tilt_beam(cpx* psi, int N, float d1, float d2, float lambda, float tb_x, float tb_y,
                      float pi, int flag, cudaStream_t st)
{
    launch(k_tilt_beam, (N * N + 255) / 256, 256, 0, st, psi, N, d1, d2, lambda, tb_x, tb_y, pi, flag);
}

// taperedCosineWindow_d, src/multisliceSimulation.cu:123-156
__global__ void k_tukey_window(cpx* psi, int N, int dn1, int dn2, float pi)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * N) return;
    const int i1 = i % N, i2 = i / N;
    float w = 1.f;
    float alpha = 2.f * (((float)dn1) / ((float)N));
    float x = ((float)i1) / ((float)(N - 1));
    if (x < alpha * 0.5f) w = 0.5f * (1.f + cosf(pi * (2.f * x / alpha - 1.f)));
    else if (x > 1.f - 0.5f * alpha) w = 0.5f * (1.f + cosf(pi * (2.f * x / alpha + 1.f - 2.f / alpha)));
    alpha = 2.f * (((float)dn2) / ((float)N));
    x = ((float)i2) / ((float)(N - 1));
    if (x < alpha * 0.5f) w *= 0.5f * (1.f + cosf(pi * (2.f * x / alpha - 1.f)));
    else if (x > 1.f - 0.5f * alpha) w *= 0.5f * (1.f + cosf(pi * (2.f * x / alpha + 1.f - 2.f / alpha)));
    psi[i] = make_float2(psi[i].x * w, psi[i].y * w);
}
void launch_tukey_window(cpx* psi, int N, int dn1, int dn2, float pi, cudaStream_t st)
{
    launch(k_tukey_window, (N * N + 255) / 256, 256, 0, st, psi, N, dn1, dn2, pi);
}

// areaMask + areaWeighting against a constant-1 field (applyMaskFiltering,
// src/crystalMaker.cu:187-224; src/multisliceSimulation.cu:468-510)
__global__ void k_area_mask_blend(cpx* psi, int N, int dn1, int dn2)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * N) return;
    const int i1 = i % N, i2 = i / N;
    float w = 1.0f;
    if (i1 <= dn1 - 1) w *= 0.5f * (1 - cosf(3.1415927f * (float)i1 / (float)dn1));
    if (i1 >= N - dn1) w *= 0.5f * (1 - cosf(3.1415927f * (float)(N - i1) / (float)dn1));
    if (i2 <= dn2 - 1) w *= 0.5f * (1 - cosf(3.1415927f * (float)i2 / (float)dn2));
    if (i2 >= N - dn2) w *= 0.5f * (1 - cosf(3.1415927f * (float)(N - i2) / (float)dn2));
    const cpx v = psi[i];
    psi[i] = make_float2(1.f * (1 - w) + v.x * w, 0.f * (1 - w) + v.y * w);
}
void launch_area_mask_blend(cpx* psi, int N, int dn1, int dn2, cudaStream_t st)
{
    launch(k_area_mask_blend, (N * N + 255) / 256, 256, 0, st, psi, N, dn1, dn2);
}

// ---------------------------------------------------------------------------------------------
// Multi-GPU reduction of the per-device partial sums (frozen-phonon configurations sharded over
// the GPUs of one process): the destination device reads the peers' buffers directly through
// NVLink peer mappings (cudaDeviceEnablePeerAccess) and adds them in the fixed order 0 .. n-1, so
// the result does not depend on timing.  128-bit loads; no staging copies.
// ---------------------------------------------------------------------------------------------
__global__ void k_peer_sum(float4* __restrict__ dst, PeerSources src, size_t n4, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        float4 a = dst[i];
        for (int r = 0; r < src.n; r++) {
            const float4 b = reinterpret_cast<const float4*>(src.p[r])[i];
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        }
        dst[i] = a;
    }
    // the last n % 4 floats (odd grid sizes)
    if (blockIdx.x == 0 && threadIdx.x < n - 4 * n4) {
        const size_t i = 4 * n4 + threadIdx.x;
        float a = reinterpret_cast<float*>(dst)[i];
        for (int r = 0; r < src.n; r++) a += src.p[r][i];
        reinterpret_cast<float*>(dst)[i] = a;
    }
}
void launch_peer_sum(float* dst, const PeerSources& src, size_t n, cudaStream_t st)
{
    const size_t n4 = n / 4;
    launch(k_peer_sum, (unsigned)std::max<size_t>(1, std::min<size_t>((n4 + 255) / 256, 148 * 8)), 256, 0, st, reinterpret_cast<float4*>(dst), src, n4, n);
}

}  // namespace fdes
