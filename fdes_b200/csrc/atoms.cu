// fdes_b200 -- atoms -> deposit records: tilt, frozen-phonon jitter, binning, stable radix sort
// and row pointers.  Replaces the per-(slice, species) full-atom scans with float atomics of the
// reference (squareAtoms_d, src/crystalMaker.cu:73-134, launched m3*nZ times per configuration)
// by ONE binning pass + ONE sort per configuration; the per-row deposits are then summed in the
// sorted (stable => deterministic) order inside the density row sweep.
#include "kernels.cuh"
#include <curand_kernel.h>   // header-only device XORWOW: same generator and seeding as the
                             // reference (curand_init / curand_normal, src/crystalMaker.cu:34,44)
#include <cfloat>
#include <cstdio>

namespace fdes {

// cublasSrot semantics used by tiltCoordinates (src/crystalMaker.cu:427-454):
// x' = c x + s y ; y' = c y - s x
__global__ void k_rot(float* xyz, int nAt, int axA, int axB, float c, float s)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nAt) return;
    const float x = xyz[3 * i + axA], y = xyz[3 * i + axB];
    xyz[3 * i + axA] = c * x + s * y;
    xyz[3 * i + axB] = c * y - s * x;
}
void launch_rot(float* xyz, int nAt, int axA, int axB, float c, float s, cudaStream_t st)
{
    launch(k_rot, (nAt + 255) / 256, 256, 0, st, xyz, nAt, axA, axB, c, s);
}

size_t rng_state_bytes() { return sizeof(curandState); }

__global__ void k_rng_init(curandState* state, int n, unsigned long long seed)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) curand_init(seed, i, 0, &state[i]);
}
void launch_rng_init(void* states, int n, unsigned long long seed, cudaStream_t st)
{
    launch(k_rng_init, (n + 127) / 128, 128, 0, st, static_cast<curandState*>(states), n, seed);
}

// atomJitter_d, src/crystalMaker.cu:37-48 (out-of-place so the equilibrium copy stays intact).
// One launch draws the displacements of `nconf` consecutive configurations: thread i advances its
// XORWOW stream by one normal per configuration, exactly like nconf successive reference launches.
__global__ void k_atom_jitter(float* __restrict__ out, const float* __restrict__ in,
                              const float* __restrict__ dwf, int nAt, curandState* state, long long burn,
                              int nconf)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * nAt) return;
    curandState local = state[i];
    for (long long b = 0; b < burn; b++) (void)curand_normal(&local);
    const float base = in[i];
    for (int c = 0; c < nconf; c++) {
        float x = curand_normal(&local);
        float v = base;
        v += x * 0.112539540f * sqrtf(dwf[i / 3]);
        out[(size_t)c * 3 * nAt + i] = v;
    }
    state[i] = local;
}
void launch_atom_jitter(float* xyz_out, const float* xyz_in, const float* dwf, int nAt,
                        void* states, long long burn, int nconf, cudaStream_t st)
{
    launch(k_atom_jitter, (3 * nAt + 127) / 128, 128, 0, st, xyz_out, xyz_in, dwf, nAt, static_cast<curandState*>(states), burn,
           nconf);
}

// ascombeNoise_d, src/crystalMaker.cu:50-70: Poisson noise via the Anscombe transform
__global__ void k_anscombe_noise(cpx* f, size_t n, float dose, curandState* state)
{
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    curandState local = state[i];
    float fi = f[i].x * dose;
    if (fi > 1e-2f) {
        float x = curand_normal(&local);
        x *= sqrtf(1 - expf(-fi / 0.777134f));
        x += 2.f * sqrtf(fi + 0.375f) - 0.25f / sqrtf(fi);
        x = roundf(0.25f * x * x - 0.375f);
        if (x < FLT_MIN) x = 0.f;
        f[i].x = x / dose;
    }
    state[i] = local;
}
void launch_anscombe_noise(cpx* f, size_t n, float dose, void* states, cudaStream_t st)
{
    launch(k_anscombe_noise, (unsigned)((n + 127) / 128), 128, 0, st, f, n, dose, static_cast<curandState*>(states));
}

// ---------------------------------------------------------------------------------------------
// binning (squareAtoms_d arithmetic, bit-exact integer indices)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int signum(float x) { return x < 0.f ? -1 : 1; }

__global__ void k_bin_atoms(const float* __restrict__ xyz, const int* __restrict__ zidx,
                            const float* __restrict__ occ, int nAt, BinGeom bg,
                            uint32_t* __restrict__ keys, int* __restrict__ cols,
                            float* __restrict__ w, int* __restrict__ bins_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nAt) return;
    // configuration blockIdx.y of a batch: coordinates [conf][nAt][3], records [conf][4 nAt]
    xyz += (size_t)blockIdx.y * 3 * nAt;
    keys += (size_t)blockIdx.y * 4 * nAt;
    cols += (size_t)blockIdx.y * 4 * nAt;
    w += (size_t)blockIdx.y * 4 * nAt;
    const int m1 = bg.m1, m2 = bg.m2, m3 = bg.m3;
    const uint32_t invalid = (uint32_t)m3 * (uint32_t)bg.nZ * (uint32_t)m2;
    const float x1 = xyz[i * 3 + 0] / bg.d1 + ((float)m1) * 0.5f - 0.5f;
    const float x2 = xyz[i * 3 + 1] / bg.d2 + ((float)m2) * 0.5f - 0.5f;
    const int i3 = (int)(roundf(xyz[i * 3 + 2] / bg.d3 + ((float)m3) * 0.5f - 0.5f));
    const bool ok = ((x1 > 1.f) && (x1 < ((float)(m1 - 2)))) && ((x2 > 1.f) && (x2 < ((float)(m2 - 2)))) &&
                    (i3 >= 0) && (i3 < m3);
    int i1 = (int)roundf(x1);
    int i2 = (int)roundf(x2);
    if (bins_out) {
        bins_out[4 * i + 0] = ok ? i1 : -1;
        bins_out[4 * i + 1] = ok ? i2 : -1;
        bins_out[4 * i + 2] = ok ? i3 : -1;
        bins_out[4 * i + 3] = zidx[i];
    }
    if (!ok) {
#pragma unroll
        for (int q = 0; q < 4; q++) { keys[4 * i + q] = invalid; cols[4 * i + q] = 0; w[4 * i + q] = 0.f; }
        return;
    }
    const float r1 = x1 - ((float)i1);
    const float r2 = x2 - ((float)i2);
    const float oc = occ[i];
    const uint32_t kbase = ((uint32_t)i3 * (uint32_t)bg.nZ + (uint32_t)zidx[i]) * (uint32_t)m2;
    // same visiting order as the reference: (i1,i2) -> (i1,i2+g2) -> (i1+g1,i2+g2) -> (i1+g1,i2)
    keys[4 * i + 0] = kbase + i2; cols[4 * i + 0] = i1;
    w[4 * i + 0] = (1 - fabsf(r1)) * (1 - fabsf(r2)) * oc;
    i2 += signum(r2);
    keys[4 * i + 1] = kbase + i2; cols[4 * i + 1] = i1;
    w[4 * i + 1] = (1 - fabsf(r1)) * fabsf(r2) * oc;
    i1 += signum(r1);
    keys[4 * i + 2] = kbase + i2; cols[4 * i + 2] = i1;
    w[4 * i + 2] = fabsf(r1) * fabsf(r2) * oc;
    i2 -= signum(r2);
    keys[4 * i + 3] = kbase + i2; cols[4 * i + 3] = i1;
    w[4 * i + 3] = fabsf(r1) * (1 - fabsf(r2)) * oc;
}

void launch_bin_atoms(const float* xyz, const int* zidx, const float* occ, int nAt,
                      const BinGeom& bg, uint32_t* keys, int* cols, float* w, int* bins_out,
                      int nconf, cudaStream_t st)
{
    launch(k_bin_atoms, dim3((nAt + 255) / 256, nconf), 256, 0, st, xyz, zidx, occ, nAt, bg, keys, cols, w, bins_out);
}

// ---------------------------------------------------------------------------------------------
// stable LSD radix sort, 8 bits per pass
// ---------------------------------------------------------------------------------------------
constexpr int SORT_THREADS = 256;
constexpr int SORT_TILES = 16;                              // tiles of 256 records per block
constexpr int SORT_CHUNK = SORT_THREADS * SORT_TILES;       // records per block

int sort_num_blocks(int n) { return n > 0 ? (n + SORT_CHUNK - 1) / SORT_CHUNK : 1; }

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_hist(const uint32_t* __restrict__ keys, int n, int shift, unsigned int* __restrict__ hist, int nb)
{
    __shared__ unsigned int h[256];
    keys += (size_t)blockIdx.y * n;
    hist += (size_t)blockIdx.y * 256 * nb;
    h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * SORT_CHUNK;
    for (int t = 0; t < SORT_TILES; t++) {
        const int i = base + t * SORT_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);   // integer counts: order-free
    }
    __syncthreads();
    hist[threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];          // digit-major
}

// exclusive scan of hist[256*nb] (digit-major) by one block
__global__ void __launch_bounds__(1024) k_sort_scan(unsigned int* hist, int total)
{
    __shared__ unsigned int sh[1024];
    hist += (size_t)blockIdx.y * total;
    const int per = (total + 1023) / 1024;
    const int lo = threadIdx.x * per, hi = min(lo + per, total);
    unsigned int s = 0;
    for (int i = lo; i < hi; i++) s += hist[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    // Hillis-Steele inclusive scan over 1024 partial sums
    for (int off = 1; off < 1024; off <<= 1) {
        unsigned int v = threadIdx.x >= off ? sh[threadIdx.x - off] : 0;
        __syncthreads();
        sh[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned int run = threadIdx.x ? sh[threadIdx.x - 1] : 0;
    for (int i = lo; i < hi; i++) { const unsigned int c = hist[i]; hist[i] = run; run += c; }
}

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_scatter(const uint32_t* __restrict__ keys, const int* __restrict__ cols,
               const float* __restrict__ w, uint32_t* __restrict__ keys_o, int* __restrict__ cols_o,
               float* __restrict__ w_o, int n, int shift, const unsigned int* __restrict__ hist, int nb)
{
    constexpr int NW = SORT_THREADS / 32;
    __shared__ unsigned int base[256];
    __shared__ unsigned int wcount[NW][256];
    {
        const size_t off = (size_t)blockIdx.y * n;
        keys += off; cols += off; w += off; keys_o += off; cols_o += off; w_o += off;
        hist += (size_t)blockIdx.y * 256 * nb;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    base[threadIdx.x] = hist[threadIdx.x * nb + blockIdx.x];
    const int cbase = blockIdx.x * SORT_CHUNK;
    for (int t = 0; t < SORT_TILES; t++) {
#pragma unroll
        for (int q = 0; q < NW; q++) wcount[q][threadIdx.x] = 0;
        __syncthreads();
        const int i = cbase + t * SORT_THREADS + threadIdx.x;
        const bool act = i < n;
        uint32_t key = 0; int col = 0; float ww = 0.f; unsigned int d = 256;
        if (act) { key = keys[i]; col = cols[i]; ww = w[i]; d = (key >> shift) & 255u; }
        // rank among equal digits inside the warp, in lane order (stable)
        const unsigned int peers = __match_any_sync(0xffffffffu, d);
        const unsigned int rank = __popc(peers & ((1u << lane) - 1u));
        if (act && rank == 0) wcount[warp][d] = __popc(peers);
        __syncthreads();
        // thread = digit: exclusive prefix over the warps, then advance the block's running base
        unsigned int run = 0;
#pragma unroll
        for (int q = 0; q < NW; q++) { const unsigned int c = wcount[q][threadIdx.x]; wcount[q][threadIdx.x] = run; run += c; }
        const unsigned int mybase = base[threadIdx.x];
        __syncthreads();
        if (act) {
            const unsigned int pos = base[d] + wcount[warp][d] + rank;
            keys_o[pos] = key; cols_o[pos] = col; w_o[pos] = ww;
        }
        __syncthreads();
        base[threadIdx.x] = mybase + run;
    }
}

void launch_radix_sort(const SortBuffers& sb, int n, int key_bits, int nconf, cudaStream_t st)
{
    if (n <= 0) return;
    const int nb = sort_num_blocks(n);
    uint32_t *ki = sb.keys, *ko = sb.keys_tmp;
    int *ci = sb.cols, *co = sb.cols_tmp;
    float *wi = sb.w, *wo = sb.w_tmp;
    int passes = (key_bits + 7) / 8;
    if (passes & 1) passes++;          // even number of passes: the result ends in the primary buffers
    if (passes == 0) passes = 2;
    for (int p = 0; p < passes; p++) {
        const int shift = 8 * p;
        launch(k_sort_hist, dim3(nb, nconf), SORT_THREADS, 0, st, ki, n, shift, sb.hist, nb);
        launch(k_sort_scan, dim3(1, nconf), 1024, 0, st, sb.hist, 256 * nb);
        launch(k_sort_scatter, dim3(nb, nconf), SORT_THREADS, 0, st, ki, ci, wi, ko, co, wo, n, shift, sb.hist, nb);
        uint32_t* tk = ki; ki = ko; ko = tk;
        int* tc = ci; ci = co; co = tc;
        float* tw2 = wi; wi = wo; wo = tw2;
    }
}

// rowptr[k] = lower_bound(keys_sorted, k)
__global__ void k_row_pointers(const uint32_t* __restrict__ keys, int n, int* __restrict__ rowptr, int nkeys, size_t rp_stride)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > nkeys) return;
    keys += (size_t)blockIdx.y * n;
    rowptr += (size_t)blockIdx.y * rp_stride;
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (keys[mid] < (uint32_t)k) lo = mid + 1; else hi = mid;
    }
    rowptr[k] = lo;
}
void launch_row_pointers(const uint32_t* keys_sorted, int n, int* rowptr, int nkeys, int nconf, cudaStream_t st, size_t rp_stride)
{
    if (rp_stride == 0) rp_stride = (size_t)nkeys + 1;
    launch(k_row_pointers, dim3((nkeys + 1 + 255) / 256, nconf), 256, 0, st, keys_sorted, n, rowptr, nkeys, rp_stride);
}

// one thread per mask word (kernels.cuh: launch_row_masks)
__global__ void k_row_masks(int* __restrict__ rowptr, size_t rp_stride, int nkeys, int N, int E)
{
    const int T = N / E, nwords = (nkeys / N) * T;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nwords) return;
    const int* rp = rowptr + (size_t)blockIdx.y * rp_stride;
    uint32_t* mask = reinterpret_cast<uint32_t*>(rowptr + (size_t)blockIdx.y * rp_stride + nkeys + 1);
    const int kg = i / T, theta = i % T;
    uint32_t w = 0;
    for (int m = 0; m < E; m++) {
        const int k = kg * N + theta + m * T;
        w |= (rp[k + 1] > rp[k] ? 1u : 0u) << m;
    }
    mask[i] = w;
}
void launch_row_masks(int* rowptr, size_t rp_stride, int nkeys, int N, int E, int nconf, cudaStream_t st)
{
    const int nwords = (nkeys / N) * (N / E);
    launch(k_row_masks, dim3((nwords + 255) / 256, nconf), 256, 0, st, rowptr, rp_stride, nkeys, N, E);
}

void launch_build_records(const float* xyz, const int* zidx, const float* occ, int nAt, const BinGeom& bg,
                          const SortBuffers& sb, int* rowptr, size_t rp_stride, int key_bits, int mask_E, int nconf,
                          cudaStream_t st)
{
    const int nrec = 4 * nAt, nkeys = bg.m3 * bg.nZ * bg.m2;
    launch_bin_atoms(xyz, zidx, occ, nAt, bg, sb.keys, sb.cols, sb.w, nullptr, nconf, st);
    launch_radix_sort(sb, nrec, key_bits, nconf, st);
    launch_row_pointers(sb.keys, nrec, rowptr, nkeys, nconf, st, rp_stride);
    if (mask_E > 0) launch_row_masks(rowptr, rp_stride, nkeys, bg.m1, mask_E, nconf, st);
}

}  // namespace fdes
