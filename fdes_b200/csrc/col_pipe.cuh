// fdes_b200 -- asynchronous column-tile pipeline for the column sweeps (S2, S4, S6) on sm_100a.
//
// A column sweep transforms every column of an [N rows][N columns] complex64 grid.  A CTA owns a
// tile of CW adjacent columns ([N][CW] elements = 64 KB at every N) and walks over tiles as a
// persistent CTA.  The tile travels between HBM/L2 and shared memory with the Tensor Memory
// Accelerator (cp.async.bulk.tensor, one elected thread issues it; SASS UTMALDG / UTMASTG), so the
// strided global loads and stores leave the instruction stream of the transform warps, and the
// load of tile i+1 and the store of tile i-1 overlap the transforms of tile i:
//
//   L   landing buffer   TMA load -> registers of the owning threads     (mbarrier `full`)
//   X   exchange buffer  Stockham passes of the line transforms          (per column, padded)
//   S   staging buffer   registers -> TMA store                          (bulk group + mbarrier `sfree`)
//
// Thread mapping: column `line` = tid / T is transformed by T = N/E consecutive threads (one warp
// for N <= 1024, 2 or 4 warps beyond: named barrier per column), thread theta holds the points
// theta + m*T, m < E -- the register layout fft_line (fft_core.cuh) expects.  The TMA box is
// [rows][CW columns] with the hardware swizzle of the row width (32/64/128 B), which spreads a
// column over 8 of the 16 eight-byte bank pairs: the per-column LDS.64/STS.64 of a warp are 2-way
// conflicted instead of 8-way for the plain dense layout.
//
// Replaces the strided cuFFT column passes of the reference (cufftExecC2C on the 2-D plan,
// src/multisliceSimulation.cu:554-556, 608-610; src/crystalMaker.cu:527-531).
#pragma once
#include "fft_core.cuh"
#include <cuda.h>
#include <cstdint>
#include <type_traits>

namespace fdes {

// ---------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier, bulk tensor copies, proxy fences
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the async proxy (TMA store source)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {}
}
// box at coordinates (x = column, y = row, z = image) of a rank-3 tensor map -> shared memory
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int x, int y, int z)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(x), "r"(y), "r"(z) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the N most recent bulk groups have finished READING their shared-memory source
template <int N_>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N_) : "memory"); }
template <int N_>
__device__ __forceinline__ void tma_store_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N_) : "memory"); }
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ---------------------------------------------------------------------------------------------
// tile geometry
// ---------------------------------------------------------------------------------------------
// Column tiles of the pipelined sweeps: 64 KB at every power-of-two N >= 512 (8192 points = 256
// threads x 32 points).
template <int N>
struct PipeCfg {
    static constexpr int E = 32;
    static constexpr int T = N / E;                       // threads per column
    static constexpr int CW = 8192 / N;                   // columns per tile: 16, 8, 4, 2
    static constexpr int THREADS = CW * T;                // 256
    static constexpr int ROWB = CW * 8;                   // bytes per tile row: 128, 64, 32, 16
    static constexpr int BR = N < 256 ? N : 256;          // rows per TMA box (box dimensions <= 256)
    static constexpr int NBOX = N / BR;
    static constexpr int TILE_BYTES = N * ROWB;           // 65536
    static constexpr int SWZ_MASK = ROWB >= 128 ? 7 : (ROWB == 64 ? 3 : (ROWB == 32 ? 1 : 0));   // CU_TENSOR_MAP_SWIZZLE_*
    static constexpr int LSTRIDE = line_smem_elems<E>(N) + 16 / CW;   // padded exchange line [elements]
    static constexpr int X_BYTES = CW * LSTRIDE * 8;
    // pass twiddle tables: copied to shared memory when they fit next to the three tile buffers (8 KB at
    // 1024, 24 KB at 2048; the 40 KB of a 4096-point line do not, they stay in global memory / L1)
    static constexpr int TW_TABLE = twiddle_table_elems<N, E>();
    static constexpr bool TW_SHARED = 2 * TILE_BYTES + ((X_BYTES + 15) & ~15) + TW_TABLE * 8 + 64 <= 227 * 1024;
    static constexpr int TW_ELEMS = TW_SHARED ? TW_TABLE : 0;
    // 1024-point columns (32 x 32): the second-pass twiddles of a thread are held in registers (TwRegs)
    static constexpr bool TW_REGS = N == 1024;
    static constexpr int OFF_L = 0, OFF_S = TILE_BYTES, OFF_X = 2 * TILE_BYTES, OFF_TW = OFF_X + ((X_BYTES + 15) & ~15),
                         OFF_BAR = OFF_TW + TW_ELEMS * 8;
    static constexpr size_t SMEM = OFF_BAR + 64;
    static constexpr bool WARP_SYNC = (T <= 32);
    // 2048-point columns as TWO 1024-point transforms, each inside one warp (see ColPipe::acquire_fft)
    static constexpr bool SPLIT = (N == 2048);
    static_assert(N >= 512 && (N & (N - 1)) == 0 && N <= 4096, "pipelined column tiles: N = 512 .. 4096, power of two");
    static_assert(T % 8 == 0, "swizzle phase of a thread must not depend on m");
};

// Synchronisation of the threads that share one column (fft_line's Sync argument).
template <int N>
struct PipeSync {
    int id;
    __device__ __forceinline__ void operator()() const
    {
        if constexpr (PipeCfg<N>::WARP_SYNC) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(PipeCfg<N>::T) : "memory");
    }
};

// Per-thread state of the pipeline.  Protocol per tile (all threads of the CTA):
//   acquire(x, next...)   wait for the landed tile, copy own points to registers, let thread 0 start
//                         the load of the next tile
//   ... transforms on x, using sm() / sync() ...
//   release(x, ...)       wait until the previous store has drained S, write own points, thread 0
//                         starts the store
// finish() before the kernel exits.
// DBG (microbenchmarks only): bit 0 = no tile loads, bit 1 = no tile stores, bit 2 = pass twiddles from
// shared memory only (no TwRegs).
template <int N, int DBG = 0>
struct ColPipe {
    using C = PipeCfg<N>;
    static constexpr bool SPLIT = C::SPLIT;
    static constexpr int E = C::E, T = C::T;
    static constexpr bool TW_REGS = C::TW_REGS && !(DBG & 4);
    unsigned char* base;       // 1024-byte aligned shared memory
    uint64_t *full, *sfree;
    const cpx* tw_global_;
    int line, theta;
    uint32_t tile_off;         // byte offset of this thread's (row theta, column line) inside a tile buffer
    uint32_t it = 0;           // tiles stored so far by this CTA
    uint32_t nload = 0;        // tiles acquired so far (several loads may feed one stored tile)
    struct NoTwRegs {};
    std::conditional_t<TW_REGS, TwRegs, NoTwRegs> twr;

    // tw: the pass twiddle tables of the line transform (global); a copy is placed in shared memory
    __device__ __forceinline__ ColPipe(unsigned char* smem_raw, const cpx* __restrict__ tw_global)
    {
        // the dynamic shared-memory array is declared __align__(1024) (swizzle atoms repeat every 1024
        // bytes); no pointer arithmetic through integers here, so that the compiler keeps the shared
        // address space (LDS / STS instead of generic LD / ST)
        base = smem_raw;
        if ((smem_u32(base) & 1023u) != 0) __trap();
        full = reinterpret_cast<uint64_t*>(base + C::OFF_BAR);
        sfree = full + 1;
        line = threadIdx.x / T;
        theta = threadIdx.x % T;
        // hardware swizzle: 16-byte chunk index ^= (byte offset >> 7) & mask; rows theta + m*T share
        // the phase of row theta because T*ROWB is a multiple of 1024
        const uint32_t o = (uint32_t)theta * C::ROWB + (uint32_t)line * 8;
        tile_off = o ^ (((o >> 7) & C::SWZ_MASK) << 4);
        if (threadIdx.x == 0) {
            mbar_init(full, 1);
            mbar_init(sfree, 1);
            fence_mbar_init();
        }
        tw_global_ = tw_global;
        cpx* tws = reinterpret_cast<cpx*>(base + C::OFF_TW);
        for (int i = threadIdx.x; i < C::TW_ELEMS; i += C::THREADS) tws[i] = tw_global[i];
        if constexpr (TW_REGS) twr.load(tw_global, theta);
        __syncthreads();
    }
    __device__ __forceinline__ auto tw() const
    {
        if constexpr (TW_REGS) return twr;
        else if constexpr (C::TW_SHARED) return TwShared{smem_u32(base + C::OFF_TW)};
        else return TwGlobal{tw_global_};
    }
    __device__ __forceinline__ cpx* sm() const { return reinterpret_cast<cpx*>(base + C::OFF_X) + line * C::LSTRIDE; }
    __device__ __forceinline__ PipeSync<N> sync() const { return PipeSync<N>{line + 1}; }

    // thread 0: start the load of the tile at column x0 of image z
    __device__ __forceinline__ void issue_load(const CUtensorMap* map, int x0, int z) const
    {
        if (DBG & 1) return;
        mbar_arrive_expect_tx(full, C::TILE_BYTES);
#pragma unroll
        for (int k = 0; k < C::NBOX; k++)
            tma_load_3d(base + C::OFF_L + k * C::BR * C::ROWB, map, full, x0, k * C::BR, z);
    }
    // x[m] <- landed tile (rows with keep(row) == false read as zero); then (have_next) thread 0
    // starts the load of the next tile
    // Keep: operator()(m): row theta + m*T is read (else zero); split(r): row lane + 32 r of a split line
    struct KeepEvery {
        __device__ __forceinline__ bool operator()(int) const { return true; }
        __device__ __forceinline__ bool split(int) const { return true; }
    };
    __device__ __forceinline__ void acquire(cpx (&x)[E], bool have_next, const CUtensorMap* map, int x0_next, int z_next)
    {
        acquire(x, have_next, map, x0_next, z_next, KeepEvery());
    }
    template <class Keep>
    __device__ __forceinline__ void acquire(cpx (&x)[E], bool have_next, const CUtensorMap* map, int x0_next, int z_next,
                                            Keep keep)
    {
        if (!(DBG & 1)) mbar_wait(full, nload & 1);
        nload++;
        const unsigned char* p = base + C::OFF_L + tile_off;
#pragma unroll
        for (int m = 0; m < E; m++) {
            const cpx v = *reinterpret_cast<const cpx*>(p + m * (T * C::ROWB));
            x[m] = keep(m) ? v : make_float2(0.f, 0.f);
        }
        __syncthreads();                       // every thread has its points: L may be overwritten
        if (threadIdx.x == 0 && have_next) issue_load(map, x0_next, z_next);
    }
    // thread 0, somewhere in the middle of a tile's work: the store of the previous tile has had
    // time to drain S; publish that to the CTA
    __device__ __forceinline__ void publish_store_drained() const
    {
        if (DBG & 2) return;
        if (threadIdx.x == 0 && it > 0) {
            tma_store_wait_read<0>();
            mbar_arrive(sfree);
        }
    }
    __device__ __forceinline__ void release(const cpx (&x)[E], const CUtensorMap* map, int x0, int z)
    {
        if (it > 0 && !(DBG & 2)) mbar_wait(sfree, (it - 1) & 1);
        unsigned char* p = base + C::OFF_S + tile_off;
#pragma unroll
        for (int m = 0; m < E; m++) *reinterpret_cast<cpx*>(p + m * (T * C::ROWB)) = x[m];
        fence_proxy_async();
        __syncthreads();
        if (threadIdx.x == 0 && !(DBG & 2)) {
#pragma unroll
            for (int k = 0; k < C::NBOX; k++)
                tma_store_3d(map, base + C::OFF_S + k * C::BR * C::ROWB, x0, k * C::BR, z);
            tma_store_commit();
        }
        it++;
    }
    __device__ __forceinline__ void finish() const
    {
        if (threadIdx.x == 0) tma_store_wait<0>();
    }

    // -----------------------------------------------------------------------------------------
    // Forward transform of the landed tile / inverse transform into the outgoing tile.
    //
    // Default: acquire + fft_line (forward), fft_line + release (inverse); x[m] <-> ky = ky0() + m*T.
    //
    // SPLIT (N = 2048, two warps w = 0, 1 per column): a radix-2 decimation step is folded into the tile
    // accesses, so that each warp runs a 1024-point transform of its own (32 x 32: ONE exchange, warp-level
    // synchronisation) instead of the two warps sharing three passes with named barriers around two
    // exchanges:
    //   forward (decimation in frequency), on the way out of the landing buffer, j = lane + 32 m < 1024:
    //       warp 0: a[j] = f[j] + f[j + 1024]                  -> X[2k]     = FFT_1024(a)[k]
    //       warp 1: b[j] = (f[j] - f[j + 1024]) W^j            -> X[2k + 1] = FFT_1024(b)[k]
    //     (each warp reads both halves of the column: 64 LDS.64 per thread, no exchange, no barrier)
    //   the spectrum is held as x[m] = X[2 (lane + 32 m) + w] = X[ky0() + m*T] with ky0() = 2 lane + w
    //   inverse (decimation in time): A = IFFT_1024(X even) in warp 0, B = IFFT_1024(X odd) in warp 1,
    //       f[j] = A[j] + conj(W)^j B[j],  f[j + 1024] = A[j] - conj(W)^j B[j]
    //     by a HALF exchange: warp 0 hands A[j], m >= 16, to warp 1 and takes conj(W)^j B[j], m < 16; each
    //     thread then writes 32 points of the outgoing tile (16 STS + 16 LDS per thread, one named barrier).
    // Per tile and thread 256 shared-memory accesses and 1 named barrier instead of 320 and 8.
    // -----------------------------------------------------------------------------------------
    static constexpr int split_tw_offset()                                   // W^j = exp(-2 pi i j / N), j < N/2
    {
        if constexpr (SPLIT) return twiddle_offset<N, E, N / 2>() + N / 2;
        else return 0;
    }
    static constexpr int SPLIT_TW = split_tw_offset();
    static constexpr int HALF_LS = line_smem_elems<E>(N / 2);               // exchange region of one warp
    __device__ __forceinline__ int ky0() const
    {
        if constexpr (SPLIT) return 2 * (theta & 31) + (theta >> 5);
        else return theta;
    }
    template <class Keep>
    __device__ __forceinline__ void acquire_fft(cpx (&x)[E], bool have_next, const CUtensorMap* map, int x0_next, int z_next,
                                                Keep keep)
    {
        if constexpr (!SPLIT) {
            acquire(x, have_next, map, x0_next, z_next, keep);
            fft_line_tw<N, E, -1>(x, sm(), theta, tw(), sync());
        } else {
            const int w = theta >> 5, lane = theta & 31;
            if (!(DBG & 1)) mbar_wait(full, nload & 1);
            nload++;
            const uint32_t o = (uint32_t)lane * C::ROWB + (uint32_t)line * 8;
            const unsigned char* p = base + C::OFF_L + (o ^ (((o >> 7) & C::SWZ_MASK) << 4));
            const auto twd = tw();
            if (w == 0) {
#pragma unroll
                for (int m = 0; m < E; m++) {
                    cpx v0 = *reinterpret_cast<const cpx*>(p + m * (32 * C::ROWB));
                    cpx v1 = *reinterpret_cast<const cpx*>(p + m * (32 * C::ROWB) + (N / 2) * C::ROWB);
                    if (!keep.split(m)) v0 = make_float2(0.f, 0.f);
                    if (!keep.split(m + E)) v1 = make_float2(0.f, 0.f);
                    x[m] = padd(v0, v1);
                }
            } else {
                split_first_odd<0>(x, p, lane, twd, keep);
            }
            __syncthreads();                       // every thread has its points: L may be overwritten
            if (threadIdx.x == 0 && have_next) issue_load(map, x0_next, z_next);
            cpx* smw = reinterpret_cast<cpx*>(base + C::OFF_X) + line * C::LSTRIDE + w * HALF_LS;
            fft_line_tw<N / 2, E, -1>(x, smw, lane, twd, SyncWarp());
        }
    }
    __device__ __forceinline__ void acquire_fft(cpx (&x)[E], bool have_next, const CUtensorMap* map, int x0_next, int z_next)
    {
        acquire_fft(x, have_next, map, x0_next, z_next, KeepEvery());
    }
    // x[M] = (f[j] - f[j + N/2]) W^j, j = lane + 32 M (compile-time table offsets)
    template <int M, class TW, class Keep>
    __device__ __forceinline__ void split_first_odd(cpx (&x)[E], const unsigned char* p, int lane, TW twd, Keep keep) const
    {
        if constexpr (M < E) {
            cpx v0 = *reinterpret_cast<const cpx*>(p + M * (32 * C::ROWB));
            cpx v1 = *reinterpret_cast<const cpx*>(p + M * (32 * C::ROWB) + (N / 2) * C::ROWB);
            if (!keep.split(M)) v0 = make_float2(0.f, 0.f);
            if (!keep.split(M + E)) v1 = make_float2(0.f, 0.f);
            x[M] = cmul(psub(v0, v1), twd.template at<SPLIT_TW + 32 * M>(lane));
            split_first_odd<M + 1>(x, p, lane, twd, keep);
        }
    }
    template <int M, class TW>
    __device__ __forceinline__ void split_last_odd(cpx (&x)[E], int lane, TW twd) const
    {
        if constexpr (M < E) {
            x[M] = cmul_conj(x[M], twd.template at<SPLIT_TW + 32 * M>(lane));
            split_last_odd<M + 1>(x, lane, twd);
        }
    }
    // inverse transform (skipped for an all-zero spectrum: do_fft = false), optional scale, and hand-over
    // of the tile
    template <bool SCALE = false>
    __device__ __forceinline__ void ifft_release(cpx (&x)[E], bool do_fft, const CUtensorMap* map, int x0, int z, float scale = 1.f)
    {
        if constexpr (!SPLIT) {
            if (do_fft) fft_line_tw<N, E, 1>(x, sm(), theta, tw(), sync());
            if constexpr (SCALE) {
#pragma unroll
                for (int m = 0; m < E; m++) x[m] = make_float2(x[m].x * scale, x[m].y * scale);
            }
            release(x, map, x0, z);
        } else {
            const int w = theta >> 5, lane = theta & 31;
            const auto twd = tw();
            cpx* col = reinterpret_cast<cpx*>(base + C::OFF_X) + line * C::LSTRIDE;
            cpx* mine = col + w * HALF_LS;
            const cpx* other = col + (1 - w) * HALF_LS;
            if (do_fft) fft_line_tw<N / 2, E, 1>(x, mine, lane, twd, SyncWarp());
            if constexpr (SCALE) {
#pragma unroll
                for (int m = 0; m < E; m++) x[m] = make_float2(x[m].x * scale, x[m].y * scale);
            }
            // the warp's own exchange region is free after its transform; the partner reads it after the
            // barrier and before the __syncthreads below, i.e. before this warp's next transform writes it
            if (w == 0) {
#pragma unroll
                for (int m = 0; m < E / 2; m++) mine[m * 32 + lane] = x[m + E / 2];
            } else {
                split_last_odd<0>(x, lane, twd);
#pragma unroll
                for (int m = 0; m < E / 2; m++) mine[m * 32 + lane] = x[m];
            }
            sync()();                              // the two warps of this column
            if (it > 0 && !(DBG & 2)) mbar_wait(sfree, (it - 1) & 1);
            const uint32_t o = (uint32_t)lane * C::ROWB + (uint32_t)line * 8;
            unsigned char* p = base + C::OFF_S + (o ^ (((o >> 7) & C::SWZ_MASK) << 4));
            if (w == 0) {
#pragma unroll
                for (int m = 0; m < E / 2; m++) {
                    const cpx b = other[m * 32 + lane];
                    *reinterpret_cast<cpx*>(p + m * (32 * C::ROWB)) = padd(x[m], b);
                    *reinterpret_cast<cpx*>(p + m * (32 * C::ROWB) + (N / 2) * C::ROWB) = psub(x[m], b);
                }
            } else {
#pragma unroll
                for (int m = E / 2; m < E; m++) {
                    const cpx a = other[(m - E / 2) * 32 + lane];
                    *reinterpret_cast<cpx*>(p + m * (32 * C::ROWB)) = padd(a, x[m]);
                    *reinterpret_cast<cpx*>(p + m * (32 * C::ROWB) + (N / 2) * C::ROWB) = psub(a, x[m]);
                }
            }
            fence_proxy_async();
            __syncthreads();
            if (threadIdx.x == 0 && !(DBG & 2)) {
#pragma unroll
                for (int k = 0; k < C::NBOX; k++)
                    tma_store_3d(map, base + C::OFF_S + k * C::BR * C::ROWB, x0, k * C::BR, z);
                tma_store_commit();
            }
            it++;
        }
    }
};

}  // namespace fdes
