// fdes_b200 -- the multislice sweeps: hand-written sm_100a kernels that replace the
// cuFFT + cuBLAS + one-thread-per-pixel chain of the reference's per-slice loop
// (phaseGrating, src/crystalMaker.cu:507-536; forwardPropagation,
// src/multisliceSimulation.cu:538-611).
//
// The wave function lives in the mixed (kx, y) domain between slices ("row space": rows are
// Fourier transformed, columns are not).  One slice is six sweeps over the grid:
//   S1 rows : density rows of each species (from sorted deposit records) -> FFT_row          -> A_z
//   S2 cols : FFT_col(A_z) * G_z, sum over species, IFFT_col                                -> B
//   S3 rows : IFFT_row(B) = V ; t0 = exp(iV) ; FFT_row(t0)                                   -> D
//   S4 cols : FFT_col(D) * (2/3 mask / N) ; IFFT_col                                         -> E
//   S5 rows : t = IFFT_row(E), psi = IFFT_row(Psi) ; FFT_row(t * psi)                        -> F
//   S6 cols : FFT_col(F) * P ; IFFT_col                                                      -> Psi'
// Every sweep reads and writes each pixel once; all multipliers come from small L2-resident
// quarter tables.  Columns that the 2/3 band limit zeroes entirely (|kx| > N/3) are neither
// stored, loaded nor transformed by S3..S6.
#pragma once
#include "fft_core.cuh"
#include "col_pipe.cuh"
#include "kernels.cuh"
#include "sweep_vtable.h"
#include <atomic>
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

namespace fdes {

// Start of every sweep launched with launch_pdl (launch.cuh): let the next sweep be scheduled, then wait until the
// previous one has finished before touching memory.
__device__ __forceinline__ void pdl_prologue()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// register budget per thread that __launch_bounds__ asks the compiler to respect
#ifndef FDES_ROW_MIN_CTAS
#define FDES_ROW_MIN_CTAS 3
#endif
#ifndef FDES_COL_MIN_CTAS
#define FDES_COL_MIN_CTAS 1
#endif

// Points per thread for a line of N points (rows and columns use the same split, so one
// twiddle table per grid size serves both).
template <int N>
struct LineCfg {
    static constexpr int E = (N & (N - 1)) != 0 ? 20                        // 2^a 5^b grids: 320, 800, 1000
                                                : (N >= 512 ? 32 : (N >= 128 ? 16 : 8));
    static constexpr int T = N / E;                     // threads per line
    static constexpr int LS = line_smem_elems<E>(N);    // padded line buffer [elements]
};
template <int N>
struct RowCfg {
    static constexpr int E = LineCfg<N>::E, T = N / E;
    static constexpr int RPB = (T & (T - 1)) != 0 ? 4 : ((128 / T) > 0 ? (128 / T) : 1);   // lines (rows) per CTA
    static constexpr int THREADS = RPB * T;
    static constexpr int LSTRIDE = line_smem_elems<E>(N);
    static constexpr size_t SMEM = (size_t)RPB * LSTRIDE * sizeof(cpx);
    static constexpr bool WARP_SYNC = (32 % T == 0);   // a line lives inside one warp
    static constexpr bool NAMED_SYNC = (T % 32 == 0);  // a line is a whole number of warps
    static constexpr int MIN_CTAS = (N >= 2048 || !WARP_SYNC) ? 2 : FDES_ROW_MIN_CTAS;   // long lines need the registers
};
// threads of one row line: warp-level sync when the line fits a warp, a named barrier when it is a
// whole number of warps, else (T = 40, 50: lines straddle warps) the whole CTA
template <int N>
struct RowSync {
    using C = RowCfg<N>;
    int id;
    __device__ __forceinline__ explicit RowSync(int line) : id(line + 1) {}
    __device__ __forceinline__ void operator()() const
    {
        if constexpr (C::WARP_SYNC) __syncwarp();
        else if constexpr (C::NAMED_SYNC) asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(C::T) : "memory");
        else __syncthreads();
    }
};
template <int N>
struct ColCfg {
    using L = LineCfg<N>;
    static constexpr int E = L::E, T = L::T;
    static constexpr int CW = (T & (T - 1)) != 0 ? (T <= 40 ? 8 : 4)                       // T = 40, 50
                                                 : ((256 / T) >= 16 ? 16 : ((256 / T) >= 2 ? (256 / T) : 2));   // columns per CTA
    static constexpr int THREADS = CW * T;
    static constexpr int LSTRIDE = L::LS + 16 / CW;   // bank-conflict-free line stride
    static constexpr size_t SMEM = (size_t)CW * LSTRIDE * sizeof(cpx);
    // Staged tiles: the CTA moves its [N rows][CW columns] tile between global and shared memory
    // with a column-fastest thread mapping (coalesced CW*8-byte row segments), while each column
    // is transformed by the threads of ONE warp (warp-level synchronisation inside the FFT).
    static constexpr bool STAGED = (32 % T == 0);
    static constexpr int RPI = THREADS / CW;          // tile rows moved per iteration (= T)
    static constexpr int MIN_CTAS = FDES_COL_MIN_CTAS;
};

template <int N>
using ColCtx = ColTile<N, LineCfg<N>::E, ColCfg<N>::CW, ColCfg<N>::STAGED>;
// Multiply x[m] (ky = theta + m*T) by the quarter table tab[ax * Q + min(ky, N - ky)] (|kx| slowest,
// |ky| fastest: the T threads of a column read consecutive entries): the first half of the points
// sits at lo + m*T, the second at hi + (N - m*T) with lo = tab + ax*Q + theta and
// hi = tab + ax*Q - theta -- compile-time offsets.
// A complex table (the propagator) is read with the evict_last L2 policy (fft_core.cuh: ld_tab_at).
// 4096^2, 34 MB table: S6 929 -> 861 us per slice of 10 images.
template <int N, int E, int M, class TabT, class F>
__device__ __forceinline__ void quarter_table_apply(cpx (&x)[E], const TabT* lo, const TabT* hi, F f)
{
    constexpr int T = N / E;
    if constexpr (M < E) {
        if constexpr (M < E / 2) x[M] = f(x[M], ld_tab_at<M * T>(lo));
        else x[M] = f(x[M], ld_tab_at<N - M * T>(hi));
        quarter_table_apply<N, E, M + 1>(x, lo, hi, f);
    }
}
struct KeepAll { __device__ __forceinline__ bool operator()(int) const { return true; } };
// Rows with deposit records, from the row-mask words of the thread's position (launch_row_masks): w0 = word of
// position theta (bit m <-> row theta + m*T); for the split lines of col_pipe.cuh w0 / w1 = words of positions
// lane / lane + 32, so that row lane + 32 r is bit r/2 of word r%2.
struct KeepMask {
    uint32_t w0, w1;
    __device__ __forceinline__ bool operator()(int m) const { return (w0 >> m) & 1u; }
    __device__ __forceinline__ bool split(int r) const { return (((r & 1) ? w1 : w0) >> (r >> 1)) & 1u; }
};
// The same rows straight from the row pointers (position pos of the line, rows pos + m*T), evaluated inside the tile
// access: 4 loads per row.  Used at 4096^2, where S2 with the mask words runs 7-25 % slower than with these
// (measured on the three-species slab, same box: 1340 us against 1440-1670 us per slice of 10 images; the L2
// hit rate of the scattering-factor tables drops from 54 % to 43 %) -- not understood, kept as measured.
struct KeepRowPtr {
    const int *rp, *rp2;
    int pos, T;
    __device__ __forceinline__ bool operator()(int m) const
    {
        const int y = pos + m * T;
        return (rp[y + 1] > rp[y]) | (rp2[y + 1] > rp2[y]);
    }
    __device__ __forceinline__ bool split(int) const { return true; }      // split lines always use the masks
};
// mask words of configuration b, key group kg = slice * nZ + z (T words each)
__device__ __forceinline__ const uint32_t* row_mask_words(const int* rowptr, size_t rp_stride, int mask_off, int b, int kg, int T)
{
    return reinterpret_cast<const uint32_t*>(rowptr + (size_t)b * rp_stride + mask_off) + (size_t)kg * T;
}

__device__ __forceinline__ bool in_band(int kx, int lo_end, int hi_start)
{
    return kx < lo_end || kx >= hi_start;
}
// band column tiles are numbered contiguously: [0, lo_end) then [hi_start, N)
__device__ __forceinline__ int band_col0(int tile_col, int lo_end, int hi_start)
{
    return tile_col < lo_end ? tile_col : hi_start + (tile_col - lo_end);
}
static int band_cols(const SweepGeom& g)
{
    return g.lo_end >= g.hi_start ? g.N : g.lo_end + (g.N - g.hi_start);
}

// The pipelined form (col_pipe.cuh): persistent CTAs, tiles fed by TMA.  Tile t covers the band
// columns [CW * ord.xt(t), +CW) of image ord.img(t) (TileOrder below).
// Tile number t of a launch -> (column tile, image): all tiles of an image first, consecutive CTAs on adjacent
// tiles (they share 128-byte lines at 16- and 32-byte tile rows).  (Visiting the same columns of all images
// together, so that a quarter-table row is fetched once per launch, was measured and gained nothing.)
struct TileOrder {
    int tiles_x;
    __device__ __forceinline__ explicit TileOrder(int tiles_x_) : tiles_x(tiles_x_) {}
    __device__ __forceinline__ int xt(int t) const { return t % tiles_x; }      // column tile
    __device__ __forceinline__ int img(int t) const { return t / tiles_x; }     // image
};

template <int N>
constexpr bool pipe_supported() { return N == 512 || N == 1024 || N == 2048 || N == 4096; }
// (N = 2048 / 4096: tile rows of 32 / 16 bytes.  With generic LD/ST, 255 registers and four-instruction
// complex multiplies the pipelined kernels were no faster than the register-staged ones there; since those
// were fixed they are 21 % / 35 % faster: tools/microbench/col_bench.cu, profiles/r2_v4_col_bench.txt)
static int pipe_grid(int ntiles)
{
    int n = pipe_cta_cap;               // (kernels.cuh) 0 unless a test asks for another tile schedule
    if (n == 0) {
        static std::atomic<int> sms[64];
        int dev = 0;
        CK(cudaGetDevice(&dev));
        n = sms[dev & 63].load();
        if (n == 0) {
            CK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
            sms[dev & 63].store(n);
        }
    }
    pipe_last_grid = ntiles < n ? ntiles : n;     // one persistent CTA per SM
    return pipe_last_grid;
}

// The reference multiplies complex fields with a 3-multiplication form (multiplyElementwise,
// src/complexMath.cu:44-62); here the plain product is used (FMUL2 + FFMA2).  Both are correctly
// rounded to within 1-2 ulp of the exact product; the parity bound is 1e-5.

// =============================================================================================
// S1  density rows
// =============================================================================================
// Two slices share one complex transform: the density of `slice` goes to the real part and the
// density of `slice2` (or nothing, slice2 < 0) to the imaginary part.  The scattering-factor
// multiplier of S2 is real and even, so the two potentials come out of S3's inverse transform as
// the real and the imaginary part -- half the potential work per slice.  (The absorptive factor
// (1 + i*imPot) of squareAtoms_d, src/crystalMaker.cu:100-119, is a constant complex scale of a
// real field and is applied in S3.)
template <int N>
__global__ void __launch_bounds__(RowCfg<N>::THREADS, RowCfg<N>::MIN_CTAS)
k_density_rows(cpx* __restrict__ A, const int* __restrict__ rowptr, const int* __restrict__ rec_col,
               const float* __restrict__ rec_w, int slice, int slice2, int nZ, size_t rec_stride,
               size_t rp_stride, int cfg_stride, int cfg_off2, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = RowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const int line = threadIdx.x / C::T, theta = threadIdx.x % C::T;
    const RowSync<N> sync(line);
    const int z = blockIdx.y, b = blockIdx.z;
    const int row = blockIdx.x * C::RPB + line;
    // image b of this launch carries slice `slice` of configuration bA (real part) and slice `slice2` of
    // configuration bB (imaginary part): bA = bB = b for a pair of consecutive slices, bA = 2b, bB = 2b + 1
    // when the odd last slices of two configurations share a transform
    const int bA = b * cfg_stride, bB = bA + cfg_off2;
    const int* rp = rowptr + (size_t)bA * rp_stride + (size_t)(slice * nZ + z) * N;
    const int lo = rp[row], hi = rp[row + 1];
    int lo2 = 0, hi2 = 0;
    if (slice2 >= 0) {
        const int* rp2 = rowptr + (size_t)bB * rp_stride + (size_t)(slice2 * nZ + z) * N;
        lo2 = rp2[row]; hi2 = rp2[row + 1];
    }
    // rows without deposits are never read by S2 (it consults the same row pointers)
    if (!__syncthreads_or(hi > lo || hi2 > lo2)) return;
    cpx* dens = smem + C::RPB * C::LSTRIDE + line * N;
#pragma unroll
    for (int m = 0; m < E; m++) dens[theta + m * C::T] = make_float2(0.f, 0.f);
    __syncthreads();
    if (theta == 0) {
        // sorted, stable order -> the summation order is fixed (deterministic, unlike the
        // float atomicAdd of squareAtoms_d, src/crystalMaker.cu:100-119)
        const int* cc = rec_col + (size_t)bA * rec_stride;
        const float* ww = rec_w + (size_t)bA * rec_stride;
        for (int i = lo; i < hi; i++) dens[cc[i]].x += ww[i];
        const int* cc2 = rec_col + (size_t)bB * rec_stride;
        const float* ww2 = rec_w + (size_t)bB * rec_stride;
        for (int i = lo2; i < hi2; i++) dens[cc2[i]].y += ww2[i];
    }
    __syncthreads();
    cpx x[E];
#pragma unroll
    for (int m = 0; m < E; m++) x[m] = dens[theta + m * C::T];
    fft_line<N, E, -1>(x, smem + line * C::LSTRIDE, theta, tw, sync);
    cpx* out = A + ((size_t)(b * nZ + z) * N + row) * N;
#pragma unroll
    for (int m = 0; m < E; m++) out[theta + m * C::T] = x[m];
}

template <int NN>
void launch_density_rows_n(const SweepGeom& g, cpx* A, const int* rowptr, const int* rec_col,
                         const float* rec_w, int slice, int slice2, int nZ, int batch, size_t rec_stride,
                         size_t rowptr_stride, int cfg_stride, int cfg_off2, cudaStream_t st)
{
    using C = RowCfg<NN>;
    const size_t smem = C::SMEM + (size_t)C::RPB * NN * sizeof(cpx);
    dim3 grid(NN / C::RPB, nZ, batch);
    launch_pdl(k_density_rows<NN>, dim3(grid), dim3(C::THREADS), smem, st, A, rowptr, rec_col, rec_w, slice, slice2, nZ,
                                                      rec_stride, rowptr_stride, cfg_stride, cfg_off2, g.tw);
}

// =============================================================================================
// S2  potential columns
// =============================================================================================
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_potential_cols(cpx* __restrict__ B, const cpx* __restrict__ A, const float* __restrict__ Gq,
                 const int* __restrict__ rowptr, int slice, int slice2, int nZ, size_t rp_stride, int mask_off,
                 int cfg_stride, int cfg_off2, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int Q = N / 2 + 1;
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = blockIdx.x * C::CW, kx = kx0 + ctx.line, b = blockIdx.y;
    const int ax = min(kx, N - kx);
    cpx acc[E];
#pragma unroll
    for (int m = 0; m < E; m++) acc[m] = make_float2(0.f, 0.f);
    bool any = false;
    for (int z = 0; z < nZ; z++) {
        const int bA = b * cfg_stride, bB = bA + cfg_off2;     // configurations of the two parts (see k_density_rows)
        const int* rp = rowptr + (size_t)bA * rp_stride + (size_t)(slice * nZ + z) * N;
        // second slice of the pair (imaginary part); the same slice again when there is none
        const int* rp2 = slice2 >= 0 ? rowptr + (size_t)bB * rp_stride + (size_t)(slice2 * nZ + z) * N : rp;
        if (rp[N] == rp[0] && rp2[N] == rp2[0]) continue;  // species absent from both slices (CTA-uniform)
        const cpx* Az = A + (size_t)(b * nZ + z) * N * N + kx0;
        cpx x[E];
        // rows without deposits were not written by S1: read them as zero
        uint32_t kw = row_mask_words(rowptr, rp_stride, mask_off, bA, slice * nZ + z, C::T)[ctx.mask_pos()];
        if (slice2 >= 0) kw |= row_mask_words(rowptr, rp_stride, mask_off, bB, slice2 * nZ + z, C::T)[ctx.mask_pos()];
        ctx.load(x, Az, KeepMask{kw, 0u}, any);
        any = true;
        fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
        const float* G = Gq + (size_t)z * Q * Q + (size_t)ax * Q;
        // acc += x * G  (tmp holds x * G; the accumulate stays a separate packed add)
        quarter_table_apply<N, E, 0>(x, G + theta, G - theta,
                                     [](cpx v, float gz) { return pmul(v, make_float2(gz, gz)); });
#pragma unroll
        for (int m = 0; m < E; m++) acc[m] = padd(acc[m], x[m]);
    }
    if (any) fft_line<N, E, 1>(acc, ctx.sm, theta, tw, ctx);
    ctx.store(acc, B + (size_t)b * N * N + kx0);
}

// Pipelined form: work items are (tile, species) pairs in the order the accumulation visits them;
// species absent from both slices of the pair are skipped (CTA-uniform test on the row pointers).
template <int N>
__global__ void __launch_bounds__(PipeCfg<N>::THREADS, 1)
k_potential_cols_tma(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                     const float* __restrict__ Gq, const int* __restrict__ rowptr, int slice, int slice2, int nZ,
                     size_t rp_stride, int mask_off, int cfg_stride, int cfg_off2, int tiles_x, int ntiles,
                     const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = PipeCfg<N>;
    extern __shared__ __align__(1024) unsigned char pipe_smem[];
    constexpr int Q = N / 2 + 1;
    constexpr int E = C::E;
    ColPipe<N> pipe(pipe_smem, tw);
    const TileOrder ord(tiles_x);
    using Pipe = ColPipe<N>;
    const int ky0 = pipe.ky0();                 // x[m] <-> ky = ky0 + m*T
    // positions of this thread's row-mask words
    const int mp0 = Pipe::SPLIT ? (pipe.theta & 31) : pipe.theta, mp1 = Pipe::SPLIT ? mp0 + 32 : mp0;
    auto rows_of = [=](int b, int z, int sl) { return rowptr + (size_t)b * rp_stride + (size_t)(sl * nZ + z) * N; };
    auto present = [=](int b, int z) {
        const int* rp = rows_of(b * cfg_stride, z, slice);
        const int* rp2 = slice2 >= 0 ? rows_of(b * cfg_stride + cfg_off2, z, slice2) : rp;
        return rp[N] != rp[0] || rp2[N] != rp2[0];
    };
    // first present species at or after (t, z), walking this CTA's tiles; t >= ntiles: none left
    auto seek = [=](int& t, int& z) {
        while (t < ntiles) {
            for (; z < nZ; z++)
                if (present(ord.img(t), z)) return;
            t += gridDim.x; z = 0;
        }
    };
    // row masks of item (tile, z): rows without deposits were not written by S1 and read as zero.  The words
    // of the NEXT item are requested before the transforms of the current one (volatile loads stay in place),
    // so their latency is not in front of the tile.
    auto load_keep = [=](int tile, int z) {
        const int bb = (ord.img(tile)) * cfg_stride;
        const uint32_t* mA = row_mask_words(rowptr, rp_stride, mask_off, bb, slice * nZ + z, C::T);
        KeepMask k{ld_nc_u32(mA + mp0), Pipe::SPLIT ? ld_nc_u32(mA + mp1) : 0u};
        if (slice2 >= 0) {
            const uint32_t* mB = row_mask_words(rowptr, rp_stride, mask_off, bb + cfg_off2, slice2 * nZ + z, C::T);
            k.w0 |= ld_nc_u32(mB + mp0);
            if (Pipe::SPLIT) k.w1 |= ld_nc_u32(mB + mp1);
        }
        return k;
    };
    int t = blockIdx.x;
    if (t >= ntiles) return;
    int lt = t, lz = 0;                       // next item to load
    seek(lt, lz);
    if (threadIdx.x == 0) {
        prefetch_tensormap(&mapA); prefetch_tensormap(&mapB);
        if (lt < ntiles) pipe.issue_load(&mapA, ord.xt(lt) * C::CW, (ord.img(lt)) * nZ + lz);
    }
    KeepMask keep_next{0u, 0u};
    if (N < 4096 && lt < ntiles) keep_next = load_keep(lt, lz);
    for (; t < ntiles; t += gridDim.x) {
        const int kx0 = ord.xt(t) * C::CW, kx = kx0 + pipe.line, b = ord.img(t);
        const int ax = min(kx, N - kx);
        cpx acc[E];
#pragma unroll
        for (int m = 0; m < E; m++) acc[m] = make_float2(0.f, 0.f);
        bool any = false;
        while (lt == t) {                      // the landed (or landing) tile belongs to this output tile
            const int z = lz;
            const KeepMask keep = keep_next;
            const int* rp = rows_of(b * cfg_stride, z, slice);
            const int* rp2 = slice2 >= 0 ? rows_of(b * cfg_stride + cfg_off2, z, slice2) : rp;
            lz++;
            seek(lt, lz);
            cpx x[E];
            if constexpr (N >= 4096) {
                pipe.acquire_fft(x, lt < ntiles, &mapA, ord.xt(lt) * C::CW, (ord.img(lt)) * nZ + lz,
                                 KeepRowPtr{rp, rp2, pipe.theta, C::T});
            } else {
                if (lt < ntiles) keep_next = load_keep(lt, lz);
                pipe.acquire_fft(x, lt < ntiles, &mapA, ord.xt(lt) * C::CW, (ord.img(lt)) * nZ + lz, keep);
            }
            any = true;
            const float* G = Gq + (size_t)z * Q * Q + (size_t)ax * Q;
            quarter_table_apply<N, E, 0>(x, G + ky0, G - ky0,
                                         [](cpx v, float gz) { return pmul(v, make_float2(gz, gz)); });
#pragma unroll
            for (int m = 0; m < E; m++) acc[m] = padd(acc[m], x[m]);
        }
        pipe.publish_store_drained();
        pipe.ifft_release(acc, any, &mapB, kx0, b);
    }
    pipe.finish();
}

template <int NN>
void launch_potential_cols_n(const SweepGeom& g, cpx* B, const cpx* A, const float* Gq,
                           const int* rowptr, int slice, int slice2, int nZ, int batch, size_t rowptr_stride,
                           int cfg_stride, int cfg_off2, cudaStream_t st)
{
    if (g.mask_off <= 0) throw std::runtime_error("S2 needs the row masks of the deposit records (SweepGeom::mask_off)");
    if constexpr (pipe_supported<NN>()) {
        using P = PipeCfg<NN>;
        const int tiles_x = NN / P::CW, ntiles = tiles_x * batch;
        CUtensorMap mapA, mapB;
        tile_map(&mapA, A, NN, batch * nZ, P::CW, P::BR);
        tile_map(&mapB, B, NN, batch, P::CW, P::BR);
        launch_pdl(k_potential_cols_tma<NN>, dim3(pipe_grid(ntiles)), dim3(P::THREADS), P::SMEM, st, mapA, mapB, Gq, rowptr, slice, slice2,
                                                                              nZ, rowptr_stride, g.mask_off, cfg_stride, cfg_off2, tiles_x, ntiles, g.tw);
    } else {
        using C = ColCfg<NN>;
        dim3 grid(NN / C::CW, batch);
        launch_pdl(k_potential_cols<NN>, dim3(grid), dim3(C::THREADS), C::SMEM, st, B, A, Gq, rowptr, slice, slice2, nZ,
                                                               rowptr_stride, g.mask_off, cfg_stride, cfg_off2, g.tw);
    }
}

// =============================================================================================
// S3  transmission rows
// =============================================================================================
// W holds the packed potential spectrum of a slice pair in the (kx, y) domain (S2); its inverse
// row transform is V_a + i V_b.  For each slice of the pair: t0 = exp(i V (1 + i imPot)) and its
// row transform goes to D[(2 b + p)], band columns only.
// sin and cos of one argument with a compact code footprint: Cody-Waite reduction to
// [-pi/4, pi/4] (three-term pi/2, exact products through FMA) and the Cephes single-precision
// minimax polynomials, ~1 ulp for |x| < 1e5.  The library sincosf() inlines its Payne-Hanek slow
// path at every call site; 64 call sites made this kernel 180 KB of code and instruction-cache
// bound.  Arguments beyond 1e5 rad (no physical potential gets there) take one shared out-of-line
// copy of the library routine.
static __device__ __noinline__ void sincos_large(float x, float* s, float* c) { sincosf(x, s, c); }
__device__ __forceinline__ void sincos_compact(float x, float& sn, float& cs)
{
    if (fabsf(x) > 1.0e5f) { sincos_large(x, &sn, &cs); return; }
    const float kf = rintf(x * 0.636619772f);
    const int k = (int)kf;
    float r = fmaf(kf, -1.57079601e+00f, x);
    r = fmaf(kf, -3.13916473e-07f, r);
    r = fmaf(kf, -5.39030253e-15f, r);
    const float r2 = r * r;
    float ps = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(ps, r2, -1.6666654611e-1f);
    ps = fmaf(ps * r2, r, r);                                   // sin(r)
    float pc = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(pc, r2, 4.166664568298827e-2f);
    pc = fmaf(pc * r2, r2, fmaf(r2, -0.5f, 1.0f));              // cos(r)
    const float a = (k & 1) ? pc : ps;                          // quadrant rotation
    const float b = (k & 1) ? ps : pc;
    sn = (k & 2) ? -a : a;
    cs = ((k + 1) & 2) ? -b : b;
}
// 2/3 band limit of a grid of size N, known at compile time: kb = largest |i1| that zeroHighFreq's
// float test keeps on the axis (src/multisliceSimulation.cu:225-250), bounds rounded outwards to
// multiples of 32 exactly as Engine::setup_tables does for SweepGeom (the launchers check that
// the two agree).  With constant bounds the per-element band tests of the unrolled row loops fold
// away (lo_end and hi_start are multiples of the thread count T of a line for N <= 2048).
template <int N>
struct Band {
    static constexpr int kb_of()
    {
        int kb = 0;
        const float mind = (float)N;
        while (kb + 1 <= N / 2 && !(((float)((kb + 1) * (kb + 1)) * 9.f / (mind * mind)) > 1.f)) kb++;
        return kb;
    }
    static constexpr int kb = kb_of();
    static constexpr int lo0 = ((kb + 1 + 31) / 32) * 32, hi0 = ((N - kb) / 32) * 32;
    static constexpr int lo_end = lo0 >= hi0 ? N : lo0, hi_start = lo0 >= hi0 ? N : hi0;
    static void check(const SweepGeom& g)
    {
        if (g.lo_end != lo_end || g.hi_start != hi_start)
            throw std::runtime_error("band limits of the sweep geometry differ from the compiled ones");
    }
};

// (cos V, sin V) = exp(iV) with packed arithmetic: Cody-Waite reduction to [-pi/4, pi/4] (the
// quadrant comes out of the mantissa of V * 2/pi + 1.5 * 2^23), the Cephes minimax polynomials of
// sincos_compact evaluated for the cosine and the sine in the two halves of one f32x2 register,
// then the rotation by the quadrant.  |V| must be below 1e5 (checked per thread by the caller).
__device__ __forceinline__ cpx expi_packed(float V)
{
    const float q = fmaf(V, 0.636619772f, 12582912.f);
    const int k = __float_as_int(q);
    const float kf = q - 12582912.f;
    float r = fmaf(kf, -1.57079601e+00f, V);
    r = fmaf(kf, -3.13916473e-07f, r);
    r = fmaf(kf, -5.39030253e-15f, r);
    const cpx rr = pmul(make_float2(r, r), make_float2(r, 1.f));                         // (r^2, r)
    const cpx r2 = make_float2(rr.x, rr.x);
    cpx u = pfma(r2, make_float2(2.443315711809948e-5f, -1.9515295891e-4f), make_float2(-1.388731625493765e-3f, 8.3321608736e-3f));
    u = pfma(u, r2, make_float2(4.166664568298827e-2f, -1.6666654611e-1f));
    u = pmul(u, r2);
    const cpx tail = pfma(rr, make_float2(-0.5f, 1.f), make_float2(1.f, 0.f));           // (1 - r^2/2, r)
    u = pfma(u, rr, tail);                                                              // (cos r, sin r)
    // rotate by k quarter turns: odd k -> (-sin, cos); k & 2 -> negate
    const bool odd = (k & 1) != 0;
    const float c0 = odd ? -u.y : u.x, s0 = odd ? u.x : u.y;
    const int sgn = (k & 2) << 30;
    return make_float2(__int_as_float(__float_as_int(c0) ^ sgn), __int_as_float(__float_as_int(s0) ^ sgn));
}
// potential2Transmission, src/multisliceSimulation.cu:41-52, with V.x = V and V.y = imPot * V; any
// argument (one out-of-line copy: only taken for |V| >= 1e5 rad, which no physical slice reaches)
static __device__ __noinline__ cpx transmission(float V, float imPot)
{
    float sn, cs;
    sincos_compact(V, sn, cs);
    if (imPot != 0.f) {
        const float e = __expf(-(V * imPot));
        return make_float2(e * cs, e * sn);
    }
    return make_float2(cs, sn);
}
// One copy of the forward line transform serves all three transforms of the sweep: the inverse
// transform of W is taken as swap(FFT(swap(W))) (real and imaginary parts exchanged on the way in
// and out), so the kernel's code is a third of the fully unrolled form and stays inside the
// instruction cache.
template <int N>
__global__ void __launch_bounds__(RowCfg<N>::THREADS, RowCfg<N>::MIN_CTAS)
k_transmit_rows(const cpx* __restrict__ W, cpx* __restrict__ D, int npair, float imPot, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = RowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    constexpr int lo_end = Band<N>::lo_end, hi_start = Band<N>::hi_start;
    const int line = threadIdx.x / C::T, theta = threadIdx.x % C::T;
    const RowSync<N> sync(line);
    const size_t row = (size_t)blockIdx.x * C::RPB + line;
    const size_t in_off = ((size_t)blockIdx.y * N + row) * N;
    cpx* sm = smem + line * C::LSTRIDE;
    float* park = reinterpret_cast<float*>(smem + C::RPB * C::LSTRIDE) + line * (2 * N);   // V_a | V_b
    cpx x[E];
#pragma unroll 1
    for (int ph = 0; ph <= npair; ph++) {
        if (ph == 0) {
#pragma unroll
            for (int m = 0; m < E; m++) {
                const cpx w = W[in_off + theta + m * C::T];
                x[m] = make_float2(w.y, w.x);
            }
        } else {
            // t0 = exp(i V (1 + i imPot)) of slice ph - 1 of the pair
            const float* V = park + (ph - 1) * N;
            float amax = 0.f;
#pragma unroll
            for (int m = 0; m < E; m++) amax = fmaxf(amax, fabsf(V[theta + m * C::T]));
            if (amax < 1.0e5f) {
#pragma unroll
                for (int m = 0; m < E; m++) {
                    const float v = V[theta + m * C::T];
                    x[m] = expi_packed(v);
                    if (imPot != 0.f) {
                        const float e = __expf(-(v * imPot));
                        x[m] = make_float2(e * x[m].x, e * x[m].y);
                    }
                }
            } else {
#pragma unroll
                for (int m = 0; m < E; m++) x[m] = transmission(V[theta + m * C::T], imPot);
            }
        }
        fft_line<N, E, -1>(x, sm, theta, tw, sync);
        if (ph == 0) {
            // IFFT_row(W) = swap(x) = V_a + i V_b
#pragma unroll
            for (int m = 0; m < E; m++) {
                park[theta + m * C::T] = x[m].y;
                park[N + theta + m * C::T] = x[m].x;
            }
        } else {
            cpx* out = D + ((size_t)(blockIdx.y * 2 + (ph - 1)) * N + row) * N;
#pragma unroll
            for (int m = 0; m < E; m++) {
                const int kx = theta + m * C::T;
                if (in_band(kx, lo_end, hi_start)) out[kx] = x[m];
            }
        }
    }
}

// ---- 2048-point rows as two 1024-point transforms, one per warp (split_dif / split_dit_combine, fft_core.cuh) ----
#ifndef FDES_SPLIT_ROWS_MIN_CTAS
#define FDES_SPLIT_ROWS_MIN_CTAS 3
#endif
template <int N>
struct SplitRowCfg {
    static constexpr int E = 32, H = N / 2, RPB = 2, THREADS = RPB * 64;
    static constexpr int HLS = line_smem_elems<E>(H);                 // exchange region of one warp
    static constexpr size_t SMEM_FFT = (size_t)RPB * 2 * HLS * sizeof(cpx);
};
struct PairSync {      // the two warps of row `line` of the CTA
    int id;
    __device__ __forceinline__ void operator()() const { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
};

// S3 for split rows: the inverse transform of W starts with the radix-2 step on the loads (no exchange), the
// forward transforms of the two transmission functions end with the half exchange.  V and t0 are held at the
// positions x = 2 (lane + 32 m) + w -- the pointwise exp(iV) does not care.
template <int N>
__global__ void __launch_bounds__(SplitRowCfg<N>::THREADS, FDES_SPLIT_ROWS_MIN_CTAS)
k_transmit_rows_split(const cpx* __restrict__ W, cpx* __restrict__ D, int npair, float imPot, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = SplitRowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    constexpr int lo_end = Band<N>::lo_end, hi_start = Band<N>::hi_start;
    const int line = threadIdx.x / 64, theta = threadIdx.x % 64, w = theta >> 5, lane = theta & 31;
    const size_t row = (size_t)blockIdx.x * C::RPB + line;
    const cpx* src = W + ((size_t)blockIdx.y * N + row) * N;
    cpx* mine = smem + (line * 2 + w) * C::HLS;
    const cpx* other = smem + (line * 2 + (1 - w)) * C::HLS;
    float* park = reinterpret_cast<float*>(smem + C::RPB * 2 * C::HLS) + line * (2 * N);   // V_a | V_b
    const TwGlobal twg{tw};
    const PairSync pair_sync{line + 1};
    cpx x[E];
#pragma unroll 1
    for (int ph = 0; ph <= npair; ph++) {
        if (ph == 0) {
            // inverse transform as swap(FFT(swap(.)))
            split_dif<N, E, -1>(x, w, lane, twg, [src](int ln, int blk) {
                const cpx v = src[ln + 32 * blk];
                return make_float2(v.y, v.x);
            });
        } else {
            const float* V = park + (ph - 1) * N;
            float amax = 0.f;
#pragma unroll
            for (int m = 0; m < E; m++) amax = fmaxf(amax, fabsf(V[theta + m * 64]));
            if (amax < 1.0e5f) {
#pragma unroll
                for (int m = 0; m < E; m++) {
                    const float v = V[theta + m * 64];
                    x[m] = expi_packed(v);
                    if (imPot != 0.f) {
                        const float e = __expf(-(v * imPot));
                        x[m] = make_float2(e * x[m].x, e * x[m].y);
                    }
                }
            } else {
#pragma unroll
                for (int m = 0; m < E; m++) x[m] = transmission(V[theta + m * 64], imPot);
            }
        }
        fft_line_tw<N / 2, E, -1>(x, mine, lane, twg, SyncWarp());
        if (ph == 0) {
#pragma unroll
            for (int m = 0; m < E; m++) {
                park[theta + m * 64] = x[m].y;
                park[N + theta + m * 64] = x[m].x;
            }
        } else {
            cpx* out = D + ((size_t)(blockIdx.y * 2 + (ph - 1)) * N + row) * N;
            split_dit_combine<N, E, -1>(x, w, lane, twg, mine, other, pair_sync, [out](int ln, int blk, cpx lo, cpx hi) {
                if (in_band(32 * blk, lo_end, hi_start)) out[ln + 32 * blk] = lo;
                if (in_band(32 * blk + N / 2, lo_end, hi_start)) out[ln + 32 * blk + N / 2] = hi;
            });
            if (ph < npair) pair_sync();      // the partner has read this warp's slots before the next transform reuses them
        }
    }
}

template <int NN>
void launch_transmit_rows_n(const SweepGeom& g, const cpx* W, cpx* D, int npair, float imPot, int batch,
                          cudaStream_t st)
{
    Band<NN>::check(g);
    if constexpr (NN == 2048) {
        using S = SplitRowCfg<NN>;
        const size_t smem = S::SMEM_FFT + (size_t)S::RPB * NN * 2 * sizeof(float);
        launch_pdl(k_transmit_rows_split<NN>, dim3(NN / S::RPB, batch), dim3(S::THREADS), smem, st, W, D, npair, imPot, g.tw);
    } else {
        using C = RowCfg<NN>;
        const size_t smem = C::SMEM + (size_t)C::RPB * NN * 2 * sizeof(float);
        dim3 grid(NN / C::RPB, batch);
        launch_pdl(k_transmit_rows<NN>, dim3(grid), dim3(C::THREADS), smem, st, W, D, npair, imPot, g.tw);
    }
}

// =============================================================================================
// S4  band-limit columns
// =============================================================================================
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, LineCfg<N>::T <= 32 ? 2 : ColCfg<N>::MIN_CTAS)
k_bandlimit_cols(cpx* __restrict__ W, int npair, int lo_end, int hi_start, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = band_col0(blockIdx.x * C::CW, lo_end, hi_start), kx = kx0 + ctx.line;
    // entry (b, p) of a [batch][2] stack; npair = 1 uses p = 0 only, npair = 0: plain [batch]
    const size_t entry = npair == 0 ? blockIdx.y : (size_t)(blockIdx.y / npair) * 2 + blockIdx.y % npair;
    cpx* tile = W + entry * N * N + kx0;
    cpx x[E];
    ctx.load(x, tile, KeepAll());
    fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
    // zeroHighFreq (src/multisliceSimulation.cu:225-250) and the 1/N of bandwidthLimit (:558-559)
    const int i1 = kx > N / 2 ? kx - N : kx;
    const float mind = (float)N;
    const float alpha = 1.f / ((float)(N * N));
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int ky = theta + m * C::T;
        const int i2 = ky > N / 2 ? ky - N : ky;
        const bool cut = ((float)(i1 * i1 + i2 * i2) * 9.f / (mind * mind)) > 1.f;
        x[m] = cut ? make_float2(0.f, 0.f) : make_float2(x[m].x * alpha, x[m].y * alpha);
    }
    fft_line<N, E, 1>(x, ctx.sm, theta, tw, ctx);
    ctx.store(x, tile);
}

template <int N>
__global__ void __launch_bounds__(PipeCfg<N>::THREADS, 1)
k_bandlimit_cols_tma(const __grid_constant__ CUtensorMap map, int npair, int lo_end, int hi_start, int tiles_x,
                     int ntiles, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = PipeCfg<N>;
    extern __shared__ __align__(1024) unsigned char pipe_smem[];
    constexpr int E = C::E;
    ColPipe<N> pipe(pipe_smem, tw);
    const TileOrder ord(tiles_x);
    const int ky0 = pipe.ky0();                 // x[m] <-> ky = ky0 + m*T
    // image y of the tile list -> entry (b, p) of a [batch][2] stack (npair = 0: plain [batch])
    auto entry = [npair](int y) { return npair == 0 ? y : (y / npair) * 2 + y % npair; };
    int t = blockIdx.x;
    if (t >= ntiles) return;
    if (threadIdx.x == 0) {
        prefetch_tensormap(&map);
        pipe.issue_load(&map, band_col0(ord.xt(t) * C::CW, lo_end, hi_start), entry(ord.img(t)));
    }
    const float mind = (float)N;
    const float alpha = 1.f / ((float)(N * N));
    for (; t < ntiles; t += gridDim.x) {
        const int kx0 = band_col0(ord.xt(t) * C::CW, lo_end, hi_start), kx = kx0 + pipe.line;
        const int tn = t + gridDim.x;
        cpx x[E];
        pipe.acquire_fft(x, tn < ntiles, &map, band_col0(ord.xt(tn) * C::CW, lo_end, hi_start), entry(ord.img(tn)));
        pipe.publish_store_drained();
        const int i1 = kx > N / 2 ? kx - N : kx;
#pragma unroll
        for (int m = 0; m < E; m++) {
            const int ky = ky0 + m * C::T;
            const int i2 = ky > N / 2 ? ky - N : ky;
            const bool cut = ((float)(i1 * i1 + i2 * i2) * 9.f / (mind * mind)) > 1.f;
            x[m] = cut ? make_float2(0.f, 0.f) : make_float2(x[m].x * alpha, x[m].y * alpha);
        }
        pipe.ifft_release(x, true, &map, kx0, entry(ord.img(t)));
    }
    pipe.finish();
}

template <int NN>
void launch_bandlimit_cols_n(const SweepGeom& g, cpx* W, int batch, int npair, cudaStream_t st)
{
    if constexpr (pipe_supported<NN>()) {
        using P = PipeCfg<NN>;
        const int nimg = npair == 0 ? batch : 2 * batch;     // images in the stack
        const int tiles_x = band_cols(g) / P::CW, ntiles = tiles_x * (npair == 0 ? batch : batch * npair);
        CUtensorMap map;
        tile_map(&map, W, NN, nimg, P::CW, P::BR);
        launch_pdl(k_bandlimit_cols_tma<NN>, dim3(pipe_grid(ntiles)), dim3(P::THREADS), P::SMEM, st, map, npair, g.lo_end, g.hi_start,
                                                                              tiles_x, ntiles, g.tw);
    } else {
        using C = ColCfg<NN>;
        dim3 grid(band_cols(g) / C::CW, npair == 0 ? batch : batch * npair);
        launch_pdl(k_bandlimit_cols<NN>, dim3(grid), dim3(C::THREADS), C::SMEM, st, W, npair, g.lo_end, g.hi_start, g.tw);
    }
}

// =============================================================================================
// S5  multiply rows
// =============================================================================================
// The three transforms (two inverse, one forward) run through ONE copy of the forward transform:
// an inverse transform is swap(FFT(swap(.))), real and imaginary parts exchanged on the way in and
// out (see k_transmit_rows).
template <int N>
__global__ void __launch_bounds__(RowCfg<N>::THREADS, RowCfg<N>::MIN_CTAS)
k_multiply_rows(cpx* __restrict__ Psi, const cpx* __restrict__ Tk, size_t e_batch_stride, int psi_full,
                const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = RowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    constexpr int lo_end = Band<N>::lo_end, hi_start = Band<N>::hi_start;
    const int line = threadIdx.x / C::T, theta = threadIdx.x % C::T;
    const RowSync<N> sync(line);
    const size_t row = (size_t)blockIdx.x * C::RPB + line;
    const cpx* e = Tk + (size_t)blockIdx.y * e_batch_stride + row * N;
    cpx* p = Psi + ((size_t)blockIdx.y * N + row) * N;
    cpx* sm = smem + line * C::LSTRIDE;
    // swap(t) = FFT(swap(Tk)) is parked in shared memory while psi is transformed (two register
    // sets of E points each would not fit)
    cpx* park = smem + C::RPB * C::LSTRIDE + line * N;
    cpx x[E];
#pragma unroll 1
    for (int ph = 0; ph < 3; ph++) {
        if (ph == 0) {
#pragma unroll
            for (int m = 0; m < E; m++) {
                const int kx = theta + m * C::T;
                const cpx v = in_band(kx, lo_end, hi_start) ? e[kx] : make_float2(0.f, 0.f);
                x[m] = make_float2(v.y, v.x);
            }
            // The psi row is needed a transform later: pull its band columns into L2 now (one 128-byte line
            // per thread and step, no registers held), so that the loads of phase 1 wait for L2, not for HBM
            // (S5 -3.4 %; prefetching the rows of a later wave as well gained nothing).
            {
                constexpr int LINES = N * 8 / 128;     // 128-byte lines of a row
                for (int l = theta; l < LINES; l += C::T) {
                    const int kx = l * 16;
                    if (psi_full || in_band(kx, lo_end, hi_start)) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + kx));
                }
            }
        } else if (ph == 1) {
            if (psi_full) {
#pragma unroll
                for (int m = 0; m < E; m++) { const cpx v = ld_g(p + theta + m * C::T); x[m] = make_float2(v.y, v.x); }
            } else {
#pragma unroll
                for (int m = 0; m < E; m++) {
                    const int kx = theta + m * C::T;
                    const cpx v = in_band(kx, lo_end, hi_start) ? ld_g(p + kx) : make_float2(0.f, 0.f);
                    x[m] = make_float2(v.y, v.x);
                }
            }
        }
        fft_line<N, E, -1>(x, sm, theta, tw, sync);
        if (ph == 0) {
#pragma unroll
            for (int m = 0; m < E; m++) park[theta + m * C::T] = x[m];
        } else if (ph == 1) {
            // t * psi from the swapped pairs: t = (a.y, a.x), psi = (b.y, b.x)
#pragma unroll
            for (int m = 0; m < E; m++) {
                const cpx a = park[theta + m * C::T], b = x[m];
                x[m] = cmul(make_float2(a.y, a.x), make_float2(b.y, b.x));
            }
        } else {
#pragma unroll
            for (int m = 0; m < E; m++) {
                const int kx = theta + m * C::T;
                if (in_band(kx, lo_end, hi_start)) p[kx] = x[m];
            }
        }
    }
}

// S5 for split rows: t = IFFT(E row) and psi = IFFT(Psi row) both start with the radix-2 step on the loads, so
// the two factors meet at the same positions x = 2 (lane + 32 m) + w; only the forward transform of the product
// needs the half exchange: one barrier of two warps per row instead of twelve.
template <int N>
__global__ void __launch_bounds__(SplitRowCfg<N>::THREADS, FDES_SPLIT_ROWS_MIN_CTAS)
k_multiply_rows_split(cpx* __restrict__ Psi, const cpx* __restrict__ Tk, size_t e_batch_stride, int psi_full,
                      const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = SplitRowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    constexpr int lo_end = Band<N>::lo_end, hi_start = Band<N>::hi_start;
    const int line = threadIdx.x / 64, theta = threadIdx.x % 64, w = theta >> 5, lane = theta & 31;
    const size_t row = (size_t)blockIdx.x * C::RPB + line;
    const cpx* e = Tk + (size_t)blockIdx.y * e_batch_stride + row * N;
    cpx* p = Psi + ((size_t)blockIdx.y * N + row) * N;
    cpx* mine = smem + (line * 2 + w) * C::HLS;
    const cpx* other = smem + (line * 2 + (1 - w)) * C::HLS;
    cpx* park = smem + C::RPB * 2 * C::HLS + line * N;
    const TwGlobal twg{tw};
    cpx x[E];
#pragma unroll 1
    for (int ph = 0; ph < 3; ph++) {
        if (ph == 0) {
            split_dif<N, E, -1>(x, w, lane, twg, [e](int ln, int blk) {
                const cpx v = in_band(32 * blk, lo_end, hi_start) ? e[ln + 32 * blk] : make_float2(0.f, 0.f);
                return make_float2(v.y, v.x);
            });
            // pull the band columns of the psi row into L2 for the next phase (see k_multiply_rows)
            constexpr int LINES = N * 8 / 128;
            for (int l = theta; l < LINES; l += 64) {
                const int kx = l * 16;
                if (psi_full || in_band(kx, lo_end, hi_start)) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + kx));
            }
        } else if (ph == 1) {
            if (psi_full) {
                split_dif<N, E, -1>(x, w, lane, twg, [p](int ln, int blk) {
                    const cpx v = ld_g(p + ln + 32 * blk);
                    return make_float2(v.y, v.x);
                });
            } else {
                split_dif<N, E, -1>(x, w, lane, twg, [p](int ln, int blk) {
                    const cpx v = in_band(32 * blk, lo_end, hi_start) ? ld_g(p + ln + 32 * blk) : make_float2(0.f, 0.f);
                    return make_float2(v.y, v.x);
                });
            }
        }
        fft_line_tw<N / 2, E, -1>(x, mine, lane, twg, SyncWarp());
        if (ph == 0) {
#pragma unroll
            for (int m = 0; m < E; m++) park[theta + m * 64] = x[m];
        } else if (ph == 1) {
#pragma unroll
            for (int m = 0; m < E; m++) {
                const cpx a = park[theta + m * 64], b = x[m];
                x[m] = cmul(make_float2(a.y, a.x), make_float2(b.y, b.x));
            }
        } else {
            split_dit_combine<N, E, -1>(x, w, lane, twg, mine, other, PairSync{line + 1}, [p](int ln, int blk, cpx lo, cpx hi) {
                if (in_band(32 * blk, lo_end, hi_start)) p[ln + 32 * blk] = lo;
                if (in_band(32 * blk + N / 2, lo_end, hi_start)) p[ln + 32 * blk + N / 2] = hi;
            });
        }
    }
}

template <int NN>
void launch_multiply_rows_n(const SweepGeom& g, cpx* Psi, const cpx* E, size_t e_batch_stride,
                          int batch, bool psi_full, cudaStream_t st)
{
    Band<NN>::check(g);
    if constexpr (NN == 2048) {
        using S = SplitRowCfg<NN>;
        const size_t smem = S::SMEM_FFT + (size_t)S::RPB * NN * sizeof(cpx);
        launch_pdl(k_multiply_rows_split<NN>, dim3(NN / S::RPB, batch), dim3(S::THREADS), smem, st, Psi, E, e_batch_stride,
                   psi_full ? 1 : 0, g.tw);
    } else {
        using C = RowCfg<NN>;
        const size_t smem = C::SMEM + (size_t)C::RPB * NN * sizeof(cpx);
        dim3 grid(NN / C::RPB, batch);
        launch_pdl(k_multiply_rows<NN>, dim3(grid), dim3(C::THREADS), smem, st, Psi, E, e_batch_stride, psi_full ? 1 : 0, g.tw);
    }
}

// =============================================================================================
// S6  propagate columns
// =============================================================================================
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_propagate_cols(cpx* __restrict__ Psi, const cpx* __restrict__ Pq, int lo_end, int hi_start,
                 const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int Q = N / 2 + 1;
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = band_col0(blockIdx.x * C::CW, lo_end, hi_start), kx = kx0 + ctx.line;
    cpx* tile = Psi + (size_t)blockIdx.y * N * N + kx0;
    cpx x[E];
    ctx.load(x, tile, KeepAll());
    fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
    const cpx* P = Pq + (size_t)min(kx, N - kx) * Q;
    quarter_table_apply<N, E, 0>(x, P + theta, P - theta, [](cpx v, cpx p) { return cmul(v, p); });
    fft_line<N, E, 1>(x, ctx.sm, theta, tw, ctx);
    ctx.store(x, tile);
}

template <int N>
__global__ void __launch_bounds__(PipeCfg<N>::THREADS, 1)
k_propagate_cols_tma(const __grid_constant__ CUtensorMap map, const __grid_constant__ CUtensorMap map_out,
                     int src_img_stride, float in_scale, const cpx* __restrict__ Pq, const cpx* __restrict__ lens,
                     int lo_end, int hi_start, int tiles_x, int ntiles, const cpx* __restrict__ tw)
{
    pdl_prologue();
    using C = PipeCfg<N>;
    extern __shared__ __align__(1024) unsigned char pipe_smem[];
    constexpr int Q = N / 2 + 1;
    constexpr int E = C::E;
    ColPipe<N> pipe(pipe_smem, tw);
    const TileOrder ord(tiles_x);
    const int ky0 = pipe.ky0();                 // x[m] <-> ky = ky0 + m*T
    int t = blockIdx.x;
    if (t >= ntiles) return;
    // image b is read from image b * src_img_stride of the source stack (in place: the same stack, stride 1)
    if (threadIdx.x == 0) {
        prefetch_tensormap(&map); prefetch_tensormap(&map_out);
        pipe.issue_load(&map, band_col0(ord.xt(t) * C::CW, lo_end, hi_start), ord.img(t) * src_img_stride);
    }
    for (; t < ntiles; t += gridDim.x) {
        const int kx0 = band_col0(ord.xt(t) * C::CW, lo_end, hi_start), kx = kx0 + pipe.line;
        const int tn = t + gridDim.x;
        cpx x[E];
        const cpx* P = Pq + (size_t)min(kx, N - kx) * Q;
        pipe.acquire_fft(x, tn < ntiles, &map, band_col0(ord.xt(tn) * C::CW, lo_end, hi_start), ord.img(tn) * src_img_stride);
        pipe.publish_store_drained();
        if (in_scale != 1.f) {
#pragma unroll
            for (int m = 0; m < E; m++) x[m] = make_float2(x[m].x * in_scale, x[m].y * in_scale);
        }
        quarter_table_apply<N, E, 0>(x, P + ky0, P - ky0, [](cpx v, cpx p) { return cmul(v, p); });
        if (lens) {
            // last slice of an imaging-mode batch: the CTF (table stored [kx][ky], as in k_ctf_cols_tma) rides on
            // the same column transform pair instead of a sweep of its own
            const cpx* tab = lens + (size_t)kx * N + ky0;
#pragma unroll
            for (int m = 0; m < E; m++) {
                const cpx w = ld_nc(tab + m * C::T);
                x[m] = make_float2(w.x * x[m].x - w.y * x[m].y, w.x * x[m].y + w.y * x[m].x);
            }
        }
        pipe.ifft_release(x, true, &map_out, kx0, ord.img(t));
    }
    pipe.finish();
}

template <int NN>
void launch_propagate_cols_n(const SweepGeom& g, cpx* Psi, const cpx* Pq, int batch, cudaStream_t st)
{
    if constexpr (pipe_supported<NN>()) {
        using P = PipeCfg<NN>;
        const int tiles_x = band_cols(g) / P::CW, ntiles = tiles_x * batch;
        CUtensorMap map;
        tile_map(&map, Psi, NN, batch, P::CW, P::BR);
        launch_pdl(k_propagate_cols_tma<NN>, dim3(pipe_grid(ntiles)), dim3(P::THREADS), P::SMEM, st, map, map, 1, 1.f, Pq,
                                                                              (const cpx*)nullptr, g.lo_end, g.hi_start, tiles_x, ntiles, g.tw);
    } else {
        using C = ColCfg<NN>;
        dim3 grid(band_cols(g) / C::CW, batch);
        launch_pdl(k_propagate_cols<NN>, dim3(grid), dim3(C::THREADS), C::SMEM, st, Psi, Pq, g.lo_end, g.hi_start, g.tw);
    }
}

// S6 reading the band columns of another image stack (launch_propagate_cols_from, kernels.cuh): pipelined kernels only
template <int NN>
void launch_propagate_cols_from_n(const SweepGeom& g, cpx* Psi, const cpx* src, int src_img_stride, int src_images, const cpx* Pq,
                                  int batch, bool times_n, const cpx* lens, cudaStream_t st)
{
    using P = PipeCfg<NN>;
    const int tiles_x = band_cols(g) / P::CW, ntiles = tiles_x * batch;
    CUtensorMap map_in, map_out;
    tile_map(&map_in, src, NN, src_images, P::CW, P::BR);
    tile_map(&map_out, Psi, NN, batch, P::CW, P::BR);
    // times_n: S5 with psi = 1 returns FFT_row(IFFT_row(D)) = N * D (unnormalised transforms): the same factor here
    launch_pdl(k_propagate_cols_tma<NN>, dim3(pipe_grid(ntiles)), dim3(P::THREADS), P::SMEM, st, map_in, map_out, src_img_stride,
               times_n ? (float)NN : 1.f, Pq, lens, g.lo_end, g.hi_start, tiles_x, ntiles, g.tw);
}

// =============================================================================================
// generic row sweep
// =============================================================================================
template <int N, int DIR, int EPI>
__global__ void __launch_bounds__(RowCfg<N>::THREADS, RowCfg<N>::MIN_CTAS)
k_rows_fft(const void* __restrict__ in_, void* __restrict__ out_, RowOpts o, int lo_end,
           int hi_start, const cpx* __restrict__ tw)
{
    using C = RowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const int line = threadIdx.x / C::T, theta = threadIdx.x % C::T;
    const RowSync<N> sync(line);
    const int y = blockIdx.x * C::RPB + line;
    const size_t rowoff = ((size_t)blockIdx.y * N + y) * N;
    cpx x[E];
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int kx = theta + m * C::T;
        if (o.in_is_real)
            x[m] = make_float2(static_cast<const float*>(in_)[rowoff + kx], 0.f);
        else if (!o.band_only_in || in_band(kx, lo_end, hi_start))
            x[m] = static_cast<const cpx*>(in_)[rowoff + kx];
        else
            x[m] = make_float2(0.f, 0.f);
    }
    fft_line<N, E, DIR>(x, smem + line * C::LSTRIDE, theta, tw, sync);
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int xx = theta + m * C::T;
        const cpx v = make_float2(x[m].x * o.scale, x[m].y * o.scale);
        if (EPI == ROW_STORE) {
            static_cast<cpx*>(out_)[rowoff + xx] =
                (o.band_only_out && !in_band(xx, lo_end, hi_start)) ? make_float2(0.f, 0.f) : v;
        } else if (EPI == ROW_ACCUM) {
            cpx* q = static_cast<cpx*>(out_) + rowoff + xx;
            const cpx old = *q;
            *q = make_float2(old.x + v.x, old.y + v.y);
        } else if (EPI == ROW_INTENS_ACCUM) {
            float* q = static_cast<float*>(out_) + rowoff + xx;
            *q += o.scale * (x[m].x * x[m].x + x[m].y * x[m].y);
        } else if (EPI == ROW_STORE_SHIFT) {
            const int ys = (y + N / 2) % N, xs = (xx + N / 2) % N;
            static_cast<cpx*>(out_)[((size_t)blockIdx.y * N + ys) * N + xs] = v;
        } else {  // ROW_CROP_REAL
            const int cx = xx - o.dn1, cy = y - o.dn2;
            if (cx >= 0 && cx < o.n1 && cy >= 0 && cy < o.n2)
                static_cast<float*>(out_)[((size_t)blockIdx.y * o.n2 + cy) * o.n1 + cx] = v.x;
        }
    }
}

template <int N, int DIR>
static void rows_fft_epi(const SweepGeom& g, const void* in, void* out, RowEpilogue epi,
                         const RowOpts& o, int batch, cudaStream_t st)
{
    using C = RowCfg<N>;
    dim3 grid(N / C::RPB, batch);
#define FDES_ROWS_CASE(EPI_)                                                                     \
    case EPI_: launch(k_rows_fft<N, DIR, EPI_>, grid, C::THREADS, C::SMEM, st, in, out, o, g.lo_end, g.hi_start, g.tw); break;
    switch (epi) {
        FDES_ROWS_CASE(ROW_STORE)
        FDES_ROWS_CASE(ROW_ACCUM)
        FDES_ROWS_CASE(ROW_INTENS_ACCUM)
        FDES_ROWS_CASE(ROW_STORE_SHIFT)
        FDES_ROWS_CASE(ROW_CROP_REAL)
    }
#undef FDES_ROWS_CASE
}

template <int NN>
void launch_rows_fft_n(const SweepGeom& g, const void* in, void* out, int dir, RowEpilogue epi,
                     const RowOpts& o, int batch, cudaStream_t st)
{
    if (dir < 0) rows_fft_epi<NN, -1>(g, in, out, epi, o, batch, st);
    else rows_fft_epi<NN, 1>(g, in, out, epi, o, batch, st);
}

// Sum over a batch in a fixed order (deterministic phonon average): for b = 0 .. nb-1 in turn,
// transform row y of in[b] and add scale * v (EPI = ROW_ACCUM, complex out) or scale * |v|^2
// (EPI = ROW_INTENS_ACCUM, float out) -- one read-modify-write of `out` per batch instead of per
// configuration.
template <int N, int DIR, int EPI>
__global__ void __launch_bounds__(RowCfg<N>::THREADS, RowCfg<N>::MIN_CTAS)
k_rows_fft_sum(const cpx* __restrict__ in, void* __restrict__ out_, RowOpts o, int nb, int lo_end,
           int hi_start, const cpx* __restrict__ tw)
{
    using C = RowCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const int line = threadIdx.x / C::T, theta = threadIdx.x % C::T;
    const RowSync<N> sync(line);
    const int y = blockIdx.x * C::RPB + line;
    const size_t rowoff = (size_t)y * N;
    cpx acc[EPI == ROW_ACCUM ? E : 1];
    float acci[EPI == ROW_ACCUM ? 1 : E];
    // start from the current content of `out`: the additions then happen in exactly the order and
    // rounding of nb successive single-configuration accumulations (results do not depend on nb)
#pragma unroll
    for (int m = 0; m < E; m++) {
    const int xx = theta + m * C::T;
    if (EPI == ROW_ACCUM) acc[m] = static_cast<const cpx*>(out_)[rowoff + xx];
    else acci[m] = static_cast<const float*>(out_)[rowoff + xx];
    }
#pragma unroll 1
    for (int b = 0; b < nb; b++) {
    const cpx* src = in + (size_t)b * N * N + rowoff;
    cpx x[E];
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int kx = theta + m * C::T;
        x[m] = (!o.band_only_in || in_band(kx, lo_end, hi_start)) ? src[kx] : make_float2(0.f, 0.f);
    }
    fft_line<N, E, DIR>(x, smem + line * C::LSTRIDE, theta, tw, sync);
    // same rounding sequence as nb successive single accumulations: out += scale * v
#pragma unroll
    for (int m = 0; m < E; m++) {
        if (EPI == ROW_ACCUM) { acc[m].x += x[m].x * o.scale; acc[m].y += x[m].y * o.scale; }   // as k_rows_fft: v = x * scale; old + v
        else acci[m] += o.scale * (x[m].x * x[m].x + x[m].y * x[m].y);
    }
    }
#pragma unroll
    for (int m = 0; m < E; m++) {
    const int xx = theta + m * C::T;
    if (EPI == ROW_ACCUM) static_cast<cpx*>(out_)[rowoff + xx] = acc[m];
    else static_cast<float*>(out_)[rowoff + xx] = acci[m];
    }
}

template <int NN>
void launch_rows_fft_sum_n(const SweepGeom& g, const cpx* in, void* out, int dir, RowEpilogue epi,
                         const RowOpts& o, int nb, cudaStream_t st)
{
    using C = RowCfg<NN>;
    dim3 grid(NN / C::RPB);
    if (dir > 0 && epi == ROW_ACCUM) {
        launch(k_rows_fft_sum<NN, 1, ROW_ACCUM>, grid, C::THREADS, C::SMEM, st, in, out, o, nb, g.lo_end, g.hi_start, g.tw);
    } else if (dir > 0 && epi == ROW_INTENS_ACCUM) {
        launch(k_rows_fft_sum<NN, 1, ROW_INTENS_ACCUM>, grid, C::THREADS, C::SMEM, st, in, out, o, nb, g.lo_end, g.hi_start, g.tw);
    } else {
        throw std::runtime_error("launch_rows_fft_sum supports inverse transforms with ROW_ACCUM / ROW_INTENS_ACCUM");
    }
}

// =============================================================================================
// generic column sweep
// =============================================================================================
template <int N, int DIR, int OP>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_cols_fft(const cpx* __restrict__ in, void* __restrict__ out_, const void* __restrict__ table,
       float scale, const cpx* __restrict__ tw)
{
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = blockIdx.x * C::CW, kx = kx0 + ctx.line;
    const size_t boff = (size_t)blockIdx.y * N * N;
    cpx x[E];
    ctx.load(x, in + boff + kx0, KeepAll());
    if (OP == COL_PLAIN) {
    fft_line<N, E, DIR>(x, ctx.sm, theta, tw, ctx);
#pragma unroll
    for (int m = 0; m < E; m++) x[m] = make_float2(x[m].x * scale, x[m].y * scale);
    ctx.store(x, static_cast<cpx*>(out_) + boff + kx0);
    return;
    }
    fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
    if (OP == COL_DP_ACCUM) {
    // |fftshift(FFT psi)|^2 / N accumulated with weight (diffractionPattern,
    // src/crystalMaker.cu:714-717; cufftShift2D_h, src/complexMath.cu:510-557)
    float* out = static_cast<float*>(out_);
    const int xs = (kx + N / 2) % N;
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int ys = (theta + m * C::T + N / 2) % N;
        out[boff + (size_t)ys * N + xs] += scale * (x[m].x * x[m].x + x[m].y * x[m].y);
    }
    return;
    }
#pragma unroll
    for (int m = 0; m < E; m++) {
    const size_t idx = (size_t)(theta + m * C::T) * N + kx;
    if (OP == COL_MUL_CPX_INV) {
        // psi * CTF as in multiplyLensFunction (src/multisliceSimulation.cu:339-340); the table is stored
        // [kx][ky], so the threads of a column read consecutive entries
        const cpx w = ld_nc(static_cast<const cpx*>(table) + (size_t)kx * N + (theta + m * C::T));
        x[m] = make_float2(w.x * x[m].x - w.y * x[m].y, w.x * x[m].y + w.y * x[m].x);
    } else {
        const float w = ld_nc(static_cast<const float*>(table) + idx);
        x[m] = make_float2(x[m].x * w, x[m].y * w);
    }
    }
    fft_line<N, E, 1>(x, ctx.sm, theta, tw, ctx);
#pragma unroll
    for (int m = 0; m < E; m++) x[m] = make_float2(x[m].x * scale, x[m].y * scale);
    ctx.store(x, static_cast<cpx*>(out_) + boff + kx0);
}

template <int N, int DIR, int OP>
static void cols_fft_one(const SweepGeom& g, const cpx* in, void* out, const void* table,
                         float scale, int batch, cudaStream_t st)
{
    using C = ColCfg<N>;
    dim3 grid(N / C::CW, batch);
    launch(k_cols_fft<N, DIR, OP>, grid, C::THREADS, C::SMEM, st, in, out, table, scale, g.tw);
}

// COL_MUL_CPX_INV on the band columns only, pipelined (col_pipe.cuh): out = scale * IFFT_col( FFT_col(in) * tab ),
// tab stored [kx][ky].  Columns outside the band are not written (the consumer reads band columns only).
template <int N>
__global__ void __launch_bounds__(PipeCfg<N>::THREADS, 1)
k_ctf_cols_tma(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_out,
               const cpx* __restrict__ table, float scale, int lo_end, int hi_start, int tiles_x, int ntiles,
               const cpx* __restrict__ tw)
{
    using C = PipeCfg<N>;
    extern __shared__ __align__(1024) unsigned char pipe_smem[];
    constexpr int E = C::E;
    ColPipe<N> pipe(pipe_smem, tw);
    const TileOrder ord(tiles_x);
    const int ky0 = pipe.ky0();                 // x[m] <-> ky = ky0 + m*T
    int t = blockIdx.x;
    if (t >= ntiles) return;
    if (threadIdx.x == 0) {
        prefetch_tensormap(&map_in); prefetch_tensormap(&map_out);
        pipe.issue_load(&map_in, band_col0(ord.xt(t) * C::CW, lo_end, hi_start), ord.img(t));
    }
    for (; t < ntiles; t += gridDim.x) {
        const int kx0 = band_col0(ord.xt(t) * C::CW, lo_end, hi_start), kx = kx0 + pipe.line;
        const int tn = t + gridDim.x;
        cpx x[E];
        pipe.acquire_fft(x, tn < ntiles, &map_in, band_col0(ord.xt(tn) * C::CW, lo_end, hi_start), ord.img(tn));
        pipe.publish_store_drained();
        const cpx* tab = table + (size_t)kx * N + ky0;
#pragma unroll
        for (int m = 0; m < E; m++) {
            const cpx w = ld_nc(tab + m * C::T);
            x[m] = make_float2(w.x * x[m].x - w.y * x[m].y, w.x * x[m].y + w.y * x[m].x);
        }
        pipe.template ifft_release<true>(x, true, &map_out, kx0, ord.img(t), scale);
    }
    pipe.finish();
}

template <int NN>
void launch_cols_fft_n(const SweepGeom& g, const cpx* in, void* out, int dir, ColOp op,
                     const void* table, float scale, int batch, cudaStream_t st)
{
    if constexpr (pipe_supported<NN>()) {
        if (op == COL_MUL_CPX_INV && g.lo_end < g.hi_start) {
            using P = PipeCfg<NN>;
            const int tiles_x = band_cols(g) / P::CW, ntiles = tiles_x * batch;
            CUtensorMap map_in, map_out;
            tile_map(&map_in, in, NN, batch, P::CW, P::BR);
            tile_map(&map_out, out, NN, batch, P::CW, P::BR);
            launch(k_ctf_cols_tma<NN>, pipe_grid(ntiles), P::THREADS, P::SMEM, st, map_in, map_out, static_cast<const cpx*>(table),
                   scale, g.lo_end, g.hi_start, tiles_x, ntiles, g.tw);
            return;
        }
    }
    switch (op) {
        case COL_PLAIN:
            if (dir < 0) cols_fft_one<NN, -1, COL_PLAIN>(g, in, out, table, scale, batch, st);
            else cols_fft_one<NN, 1, COL_PLAIN>(g, in, out, table, scale, batch, st);
            break;
        case COL_MUL_CPX_INV: cols_fft_one<NN, -1, COL_MUL_CPX_INV>(g, in, out, table, scale, batch, st); break;
        case COL_MUL_REAL_INV: cols_fft_one<NN, -1, COL_MUL_REAL_INV>(g, in, out, table, scale, batch, st); break;
        case COL_DP_ACCUM: cols_fft_one<NN, -1, COL_DP_ACCUM>(g, in, out, table, scale, batch, st); break;
    }
}

// =============================================================================================
// STEM: shifted probes from the spectrum of the centred probe, and annular detectors
// =============================================================================================
// Psi_b(kx, y) = (1/N) IFFT_col[ PSI0(kx, ky) * exp(-2 pi i (iw(kx) sx_b + iw(ky) sy_b)) ], band
// columns only; PSI0 = FFT_col of the centred, normalised probe in the (kx, y) domain.  shifts:
// [batch][2] = probe position / (N * pixel size), i.e. in units of the grid period.
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_probe_cols(cpx* __restrict__ Psi, const cpx* __restrict__ PSI0, const float* __restrict__ shifts,
             int lo_end, int hi_start, const cpx* __restrict__ tw)
{
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = band_col0(blockIdx.x * C::CW, lo_end, hi_start), kx = kx0 + ctx.line;
    const float sx = shifts[2 * blockIdx.y], sy = shifts[2 * blockIdx.y + 1];
    cpx x[E];
    ctx.load(x, PSI0 + kx0, KeepAll());
    const int i1 = kx > N / 2 ? kx - N : kx;
    // phase in turns: the fractional part of each product is taken exactly (one rounding) before they are added,
    // so the error stays near 1e-7 turns at any N instead of growing with |i sx|
    const float ax = fmaf((float)i1, sx, -rintf((float)i1 * sx));
    const float inv = 1.f / (float)N;
#pragma unroll
    for (int m = 0; m < E; m++) {
    const int ky = theta + m * C::T;
    const int i2 = ky > N / 2 ? ky - N : ky;
    float t = ax + fmaf((float)i2, sy, -rintf((float)i2 * sy));
    t -= rintf(t);
    float sn, cs;
    sincos_compact(-6.283185307179586f * t, sn, cs);
    x[m] = cmul(x[m], make_float2(cs * inv, sn * inv));
    }
    fft_line<N, E, 1>(x, ctx.sm, theta, tw, ctx);
    ctx.store(x, Psi + (size_t)blockIdx.y * N * N + kx0);
}

template <int NN>
void launch_probe_cols_n(const SweepGeom& g, cpx* Psi, const cpx* PSI0, const float* shifts, int batch,
                       cudaStream_t st)
{
    using C = ColCfg<NN>;
    dim3 grid(band_cols(g) / C::CW, batch);
    launch(k_probe_cols<NN>, grid, C::THREADS, C::SMEM, st, Psi, PSI0, shifts, g.lo_end, g.hi_start, g.tw);
}

// partial[b][tile][d] = sum over the tile's columns and all ky of |FFT_col(Psi_b)|^2 inside the
// annulus k_in^2 <= |k|^2 < k_out^2 of detector d (|FFT2 psi|^2 / N^2 with Psi = FFT_row(psi)/N,
// the normalisation of diffractionPattern, src/crystalMaker.cu:714-717).  Fixed reduction order.
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_detector_cols(const cpx* __restrict__ Psi, float* __restrict__ partial, DetectorRings rings, float inv_l1,
                float inv_l2, int lo_end, int hi_start, const cpx* __restrict__ tw)
{
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E;
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    const int kx0 = band_col0(blockIdx.x * C::CW, lo_end, hi_start), kx = kx0 + ctx.line;
    cpx x[E];
    ctx.load(x, Psi + (size_t)blockIdx.y * N * N + kx0, KeepAll());
    fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
    const int i1 = kx > N / 2 ? kx - N : kx;
    const float k1 = (float)i1 * inv_l1;
    float acc[MAX_DETECTORS];
#pragma unroll
    for (int d = 0; d < MAX_DETECTORS; d++) acc[d] = 0.f;
#pragma unroll
    for (int m = 0; m < E; m++) {
        const int ky = theta + m * C::T;
        const int i2 = ky > N / 2 ? ky - N : ky;
        const float k2v = (float)i2 * inv_l2;
        const float ksq = k1 * k1 + k2v * k2v;
        const float v = x[m].x * x[m].x + x[m].y * x[m].y;
#pragma unroll
        for (int d = 0; d < MAX_DETECTORS; d++)
            if (d < rings.n && ksq >= rings.in2[d] && ksq < rings.out2[d]) acc[d] += v;
    }
    // deterministic CTA reduction: thread order within shared memory, then a serial sum
    __syncthreads();
    float* red = reinterpret_cast<float*>(smem);
    for (int d = 0; d < rings.n; d++) {
        red[threadIdx.x] = acc[d];
        __syncthreads();
        // ceil-halving tree: correct for any thread count (320 and 200 threads at N = 800, 1000)
        for (int n = C::THREADS; n > 1;) {
            const int s = (n + 1) / 2;
            if ((int)threadIdx.x + s < n) red[threadIdx.x] += red[threadIdx.x + s];
            __syncthreads();
            n = s;
        }
        if (threadIdx.x == 0) partial[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * MAX_DETECTORS + d] = red[0];
        __syncthreads();
    }
}

// out[b][d] += weight * sum_tiles partial[b][tile][d]
static __global__ void k_detector_finish(const float* __restrict__ partial, float* __restrict__ out, int ntiles, int ndet,
                                  int batch, float weight)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch * ndet) return;
    const int b = i / ndet, d = i % ndet;
    float s = 0.f;
    for (int t = 0; t < ntiles; t++) s += partial[((size_t)b * ntiles + t) * MAX_DETECTORS + d];
    out[(size_t)b * ndet + d] += weight * s;
}

template <int NN>
int detector_tiles_n(const SweepGeom& g)
{
    return band_cols(g) / ColCfg<NN>::CW;
}

template <int NN>
void launch_detector_cols_n(const SweepGeom& g, const cpx* Psi, float* partial, float* out, const DetectorRings& rings,
                          float d1, float d2, float weight, int batch, cudaStream_t st)
{
    using C = ColCfg<NN>;
    const int tiles = band_cols(g) / C::CW;
    dim3 grid(tiles, batch);
    launch(k_detector_cols<NN>, grid, C::THREADS, C::SMEM, st, Psi, partial, rings, 1.f / ((float)NN * d1), 1.f / ((float)NN * d2),
           g.lo_end, g.hi_start, g.tw);
    const int n = batch * rings.n;
    launch(k_detector_finish, (n + 127) / 128, 128, 0, st, partial, out, tiles, rings.n, batch, weight);
}

// 4D-STEM: scratch[b][qy][qx] = |FFT_col(Psi_b)|^2 at the window pixel (qy, qx) of the fftshifted pattern, for the
// band columns inside the window [o, o + Q)^2, o = (N - Q) / 2 (the other pixels are not written).  A thread holds
// rows ky = theta + m*T of one column; the CTA's [N][CW] intensities go through shared memory, so that each
// window row is stored as CW consecutive floats.
template <int N>
__global__ void __launch_bounds__(ColCfg<N>::THREADS, ColCfg<N>::MIN_CTAS)
k_detector4d_cols(const cpx* __restrict__ Psi, float* __restrict__ scratch, int Q, int lo_end, int hi_start,
                  const cpx* __restrict__ tw)
{
    using C = ColCfg<N>;
    extern __shared__ cpx smem[];
    constexpr int E = C::E, CWP = C::CW + 1;     // odd row stride: the T rows of a column hit distinct banks
    const int o = (N - Q) / 2;
    const int kx0 = band_col0(blockIdx.x * C::CW, lo_end, hi_start);
    bool any = false;
    for (int l = 0; l < C::CW; l++) any |= (unsigned)((kx0 + l + N / 2) % N - o) < (unsigned)Q;
    if (!any) return;                              // no column of this tile inside the window (CTA-uniform)
    const ColCtx<N> ctx(smem);
    const int theta = ctx.theta;
    cpx x[E];
    ctx.load(x, Psi + (size_t)blockIdx.y * N * N + kx0, KeepAll());
    fft_line<N, E, -1>(x, ctx.sm, theta, tw, ctx);
    __syncthreads();
    float* st = reinterpret_cast<float*>(smem);
#pragma unroll
    for (int m = 0; m < E; m++) st[(theta + m * C::T) * CWP + ctx.line] = x[m].x * x[m].x + x[m].y * x[m].y;
    __syncthreads();
    float* out = scratch + (size_t)blockIdx.y * Q * Q;
    for (int w = threadIdx.x; w < Q * C::CW; w += C::THREADS) {
        const int qy = w / C::CW, l = w % C::CW;
        const int qx = (kx0 + l + N / 2) % N - o;
        const int ky = (qy + o + N - N / 2) % N;  // inverse of the shift (ky + N/2) % N
        if ((unsigned)qx < (unsigned)Q) out[(size_t)qy * Q + qx] = st[ky * CWP + l];
    }
}

template <int NN>
void launch_detector4d_cols_n(const SweepGeom& g, const cpx* Psi, float* scratch, float* out, int Q, int bin, float weight,
                              int batch, cudaStream_t st)
{
    using C = ColCfg<NN>;
    static_assert((size_t)NN * (C::CW + 1) * sizeof(float) <= C::SMEM, "intensity tile must fit the line buffers");
    dim3 grid(band_cols(g) / C::CW, batch);
    launch(k_detector4d_cols<NN>, grid, C::THREADS, C::SMEM, st, Psi, scratch, Q, g.lo_end, g.hi_start, g.tw);
    launch_detector4d_finish(scratch, out, Q, bin, weight, batch, st);
}

// ---------------------------------------------------------------------------------------------
// twiddle tables (layout: fft_core.cuh) and geometry queries
// ---------------------------------------------------------------------------------------------
// pass twiddle tables of a line of N points with E points per thread, appended to tw
template <int N, int E>
void append_twiddles(std::vector<cpx>& tw)
{
    const size_t before = tw.size();
    int NS = 1;
    while (NS < N) {
        const int rem = N / NS, R = pass_radix(rem, E);
        if (NS > 1)
            for (int t = 0; t < R; t++)
                for (int k = 0; k < NS; k++) {
                    // exp(-2 pi i t k / (NS R)), exact on the axes
                    const long long num = (long long)t * k, den = (long long)NS * R;
                    const long long r = num % den;
                    cpx w;
                    if (r == 0) w = make_float2(1.f, 0.f);
                    else if (4 * r == den) w = make_float2(0.f, -1.f);
                    else if (2 * r == den) w = make_float2(-1.f, 0.f);
                    else if (4 * r == 3 * den) w = make_float2(0.f, 1.f);
                    else {
                        const double a = -2.0 * 3.14159265358979323846 * (double)r / (double)den;
                        w = make_float2((float)cos(a), (float)sin(a));
                    }
                    tw.push_back(w);
                }
        NS *= R;
    }
    if ((int)(tw.size() - before) != twiddle_table_elems<N, E>()) throw std::runtime_error("twiddle table size mismatch");
}
// The table a SweepGeom::tw of size N points to: the one of LineCfg<N>::E.
template <int N>
std::vector<cpx> make_twiddles_n(int = 0)
{
    std::vector<cpx> tw;
    append_twiddles<N, LineCfg<N>::E>(tw);
    if (tw.empty()) tw.push_back(make_float2(1.f, 0.f));
    return tw;
}

// S6 from another image stack exists where the column sweeps are pipelined
template <int N>
constexpr decltype(SweepVTable::propagate_cols_from) propagate_cols_from_entry()
{
    if constexpr (pipe_supported<N>()) return &launch_propagate_cols_from_n<N>;
    else return nullptr;
}

// the launchers of one grid size, collected for the run-time dispatch in sweeps.cu
template <int N>
const SweepVTable* make_sweep_vtable()
{
    static const SweepVTable vt = {
        N, RowCfg<N>::RPB, ColCfg<N>::CW, LineCfg<N>::E,
        &launch_density_rows_n<N>, &launch_potential_cols_n<N>, &launch_transmit_rows_n<N>,
        &launch_bandlimit_cols_n<N>, &launch_multiply_rows_n<N>, &launch_propagate_cols_n<N>,
        &launch_rows_fft_n<N>, &launch_rows_fft_sum_n<N>, &launch_cols_fft_n<N>,
        &launch_probe_cols_n<N>, &detector_tiles_n<N>, &launch_detector_cols_n<N>, &launch_detector4d_cols_n<N>,
        &make_twiddles_n<N>, propagate_cols_from_entry<N>(), pipe_supported<N>(),
    };
    return &vt;
}

}  // namespace fdes
