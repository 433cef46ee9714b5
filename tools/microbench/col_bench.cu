// Developer microbenchmark: the register-staged column sweep S6 (k_propagate_cols) against the
// TMA-pipelined persistent form (k_propagate_cols_tma, col_pipe.cuh) on random data; the two must
// agree bit for bit (same arithmetic, different data movement).  run_tw_ab: pass twiddles of the
// pipelined form in registers against shared memory.
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -I ../../fdes_b200/csrc col_bench.cu ../../fdes_b200/csrc/tma_map.cu -o col_bench
#include "sweep_kernels.cuh"
#include <algorithm>
#include <array>
#include <cstring>
using namespace fdes;

// copy of k_propagate_cols_tma with the debug switches of ColPipe and per-CTA cycle counters:
// dbg[cta] = {total, waiting for the landed tile, waiting for the previous store to drain, release}
template <int N, int DBG>
__global__ void __launch_bounds__(PipeCfg<N>::THREADS, 1)
k_dbg(const __grid_constant__ CUtensorMap map, const cpx* __restrict__ Pq, int lo_end, int hi_start,
      int tiles_x, int ntiles, const cpx* __restrict__ tw, long long* dbg)
{
    using C = PipeCfg<N>;
    extern __shared__ __align__(1024) unsigned char pipe_smem[];
    constexpr int Q = N / 2 + 1;
    constexpr int E = C::E;
    ColPipe<N, DBG> pipe(pipe_smem, tw);
    const int theta = pipe.ky0();
    int t = blockIdx.x;
    if (t >= ntiles) return;
    long long c_full = 0, c_drain = 0, c_rel = 0;
    const long long c_start = clock64();
    if (threadIdx.x == 0) pipe.issue_load(&map, band_col0((t % tiles_x) * C::CW, lo_end, hi_start), t / tiles_x);
    for (; t < ntiles; t += gridDim.x) {
        const int kx0 = band_col0((t % tiles_x) * C::CW, lo_end, hi_start), kx = kx0 + pipe.line;
        const int tn = t + gridDim.x;
        cpx x[E];
        long long c0 = clock64();
        if (!(DBG & 1)) mbar_wait(pipe.full, pipe.nload & 1);
        c_full += clock64() - c0;
        pipe.acquire_fft(x, tn < ntiles, &map, band_col0((tn % tiles_x) * C::CW, lo_end, hi_start), tn / tiles_x);
        c0 = clock64();
        pipe.publish_store_drained();
        c_drain += clock64() - c0;
        const cpx* P = Pq + (size_t)min(kx, N - kx) * Q;
        quarter_table_apply<N, E, 0>(x, P + theta, P - theta, [](cpx v, cpx p) { return cmul(v, p); });
        c0 = clock64();
        pipe.ifft_release(x, true, &map, kx0, t / tiles_x);      // inverse transform + hand-over
        c_rel += clock64() - c0;
    }
    pipe.finish();
    if (threadIdx.x == 0 && dbg) {
        dbg[4 * blockIdx.x + 0] = clock64() - c_start;
        dbg[4 * blockIdx.x + 1] = c_full;
        dbg[4 * blockIdx.x + 2] = c_drain;
        dbg[4 * blockIdx.x + 3] = c_rel;
    }
}

template <int N, int DBG>
void run_dbg(int batch, int reps)
{
    const size_t NN = (size_t)N * N, total = NN * batch, Q = N / 2 + 1;
    cpx *d1, *P, *tw; long long* dbg;
    CK(cudaMalloc(&d1, total * sizeof(cpx))); CK(cudaMalloc(&P, Q * Q * sizeof(cpx))); CK(cudaMalloc(&dbg, 4 * 148 * sizeof(long long)));
    CK(cudaMemset(d1, 0, total * sizeof(cpx))); CK(cudaMemset(P, 0, Q * Q * sizeof(cpx)));
    auto twh = make_twiddles_n<N>();
    CK(cudaMalloc(&tw, twh.size() * sizeof(cpx)));
    CK(cudaMemcpy(tw, twh.data(), twh.size() * sizeof(cpx), cudaMemcpyHostToDevice));
    SweepGeom g{N, Band<N>::lo_end, Band<N>::hi_start, tw};
    using Pc = PipeCfg<N>;
    CK(cudaFuncSetAttribute(k_dbg<N, DBG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Pc::SMEM));
    const int bc = band_cols(g), tiles_x = bc / Pc::CW, ntiles = tiles_x * batch;
    CUtensorMap mapv; tile_map(&mapv, d1, N, batch, Pc::CW, Pc::BR); const CUtensorMap* map = &mapv;
    const int grid1 = ntiles < 148 ? ntiles : 148;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float ms1 = 0;
    for (int w = 0; w < 2; w++) {
        cudaEventRecord(e0);
        for (int r = 0; r < reps; r++) k_dbg<N, DBG><<<grid1, Pc::THREADS, Pc::SMEM>>>(*map, P, g.lo_end, g.hi_start, tiles_x, ntiles, tw, dbg);
        cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms1, e0, e1);
    }
    CK(cudaDeviceSynchronize());
    std::vector<long long> hd(4 * 148);
    CK(cudaMemcpy(hd.data(), dbg, hd.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    double s[4] = {0, 0, 0, 0};
    for (int c = 0; c < grid1; c++) for (int k = 0; k < 4; k++) s[k] += (double)hd[4 * c + k] / grid1;
    printf("N=%4d batch=%2d DBG=%d (1: no loads, 2: no stores): %8.2f us | mean cycles per CTA: total %.0f, wait-landed %.0f, wait-drain %.0f, release %.0f (tiles per CTA %.2f)\n",
           N, batch, DBG, ms1 / reps * 1e3, s[0], s[1], s[2], s[3], (double)ntiles / grid1);
    cudaFree(d1); cudaFree(P); cudaFree(tw); cudaFree(dbg);
}

template <int N>
void run(int batch, int reps)
{
    const size_t NN = (size_t)N * N, total = NN * batch, Q = N / 2 + 1;
    std::vector<cpx> h(total), ph(Q * Q);
    srand(1234);
    for (auto& v : h) v = make_float2(rand() / (float)RAND_MAX - 0.5f, rand() / (float)RAND_MAX - 0.5f);
    for (size_t i = 0; i < Q * Q; i++) { const float a = 0.001f * (float)(i % 977); ph[i] = make_float2(cosf(a) / N, sinf(a) / N); }
    cpx *d0, *d1, *P, *tw;
    CK(cudaMalloc(&d0, total * sizeof(cpx))); CK(cudaMalloc(&d1, total * sizeof(cpx))); CK(cudaMalloc(&P, Q * Q * sizeof(cpx)));
    auto twh = make_twiddles_n<N>();
    CK(cudaMalloc(&tw, twh.size() * sizeof(cpx)));
    CK(cudaMemcpy(tw, twh.data(), twh.size() * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(P, ph.data(), Q * Q * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d0, h.data(), total * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d1, h.data(), total * sizeof(cpx), cudaMemcpyHostToDevice));
    // 2/3 band limit bounds as in make_sweep_geom (sweeps.cu)
    SweepGeom g{N, Band<N>::lo_end, Band<N>::hi_start, tw};
    using C = ColCfg<N>;
    using Pc = PipeCfg<N>;
    CK(cudaFuncSetAttribute(k_propagate_cols<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    CK(cudaFuncSetAttribute(k_propagate_cols_tma<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Pc::SMEM));
    const int bc = band_cols(g);
    dim3 grid0(bc / C::CW, batch);
    const int tiles_x = bc / Pc::CW, ntiles = tiles_x * batch;
    CUtensorMap mapv; tile_map(&mapv, d1, N, batch, Pc::CW, Pc::BR); const CUtensorMap* map = &mapv;
    int nsm = 0; CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, 0));
    const int grid1 = ntiles < nsm ? ntiles : nsm;
    k_propagate_cols<N><<<grid0, C::THREADS, C::SMEM>>>(d0, P, g.lo_end, g.hi_start, tw);
    CK(cudaGetLastError());
    k_propagate_cols_tma<N><<<grid1, Pc::THREADS, Pc::SMEM>>>(*map, *map, 1, 1.f, P, (const cpx*)nullptr, g.lo_end, g.hi_start, tiles_x, ntiles, tw);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<cpx> a(total), b(total);
    CK(cudaMemcpy(a.data(), d0, total * sizeof(cpx), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b.data(), d1, total * sizeof(cpx), cudaMemcpyDeviceToHost));
    size_t diff = 0, changed = 0;
    double num = 0, den = 0;
    for (size_t i = 0; i < total; i++) {
        diff += memcmp(&a[i], &b[i], sizeof(cpx)) != 0; changed += memcmp(&a[i], &h[i], sizeof(cpx)) != 0;
        num += (double)(a[i].x - b[i].x) * (a[i].x - b[i].x) + (double)(a[i].y - b[i].y) * (a[i].y - b[i].y);
        den += (double)a[i].x * a[i].x + (double)a[i].y * a[i].y;
    }
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float ms0 = 0, ms1 = 0;
    for (int w = 0; w < 2; w++) {
        cudaEventRecord(e0);
        for (int r = 0; r < reps; r++) k_propagate_cols<N><<<grid0, C::THREADS, C::SMEM>>>(d0, P, g.lo_end, g.hi_start, tw);
        cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms0, e0, e1);
        cudaEventRecord(e0);
        for (int r = 0; r < reps; r++) k_propagate_cols_tma<N><<<grid1, Pc::THREADS, Pc::SMEM>>>(*map, *map, 1, 1.f, P, (const cpx*)nullptr, g.lo_end, g.hi_start, tiles_x, ntiles, tw);
        cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms1, e0, e1);
    }
    CK(cudaDeviceSynchronize());
    cudaFuncAttributes f0, f1;
    cudaFuncGetAttributes(&f0, k_propagate_cols<N>); cudaFuncGetAttributes(&f1, k_propagate_cols_tma<N>);
    const double gb = 16.0 * total / 1e9;
    printf("N=%4d batch=%2d band=%4d | staged CW=%2d regs=%3d: %8.2f us %6.0f GB/s | tma CW=%2d regs=%3d grid=%d tiles=%d: %8.2f us %6.0f GB/s | differing=%zu changed=%zu of %zu rel-L2 %.2e\n",
           N, batch, bc, C::CW, f0.numRegs, ms0 / reps * 1e3, gb / (ms0 / reps * 1e-3), Pc::CW, f1.numRegs, grid1, ntiles,
           ms1 / reps * 1e3, gb / (ms1 / reps * 1e-3), diff, changed, total, sqrt(num / (den > 0 ? den : 1)));
    cudaFree(d0); cudaFree(d1); cudaFree(P); cudaFree(tw);
}

// A/B of ColPipe's pass twiddles at N: registers (TwRegs, DBG 0) against shared memory only (DBG 4), in
// k_dbg (the S6 kernel), `rounds` alternated timings of `reps` launches each on the same random stack of
// `batch` images; the two outputs of one launch on the same input must agree bit for bit.
template <int N>
void run_tw_ab(int batch, int reps, int rounds)
{
    const size_t NN = (size_t)N * N, total = NN * batch, Q = N / 2 + 1;
    std::vector<cpx> h(total), ph(Q * Q);
    srand(4321);
    for (auto& v : h) v = make_float2(rand() / (float)RAND_MAX - 0.5f, rand() / (float)RAND_MAX - 0.5f);
    for (size_t i = 0; i < Q * Q; i++) { const float a = 0.001f * (float)(i % 977); ph[i] = make_float2(cosf(a) / N, sinf(a) / N); }
    cpx *da, *db, *P, *tw;
    CK(cudaMalloc(&da, total * sizeof(cpx))); CK(cudaMalloc(&db, total * sizeof(cpx))); CK(cudaMalloc(&P, Q * Q * sizeof(cpx)));
    auto twh = make_twiddles_n<N>();
    CK(cudaMalloc(&tw, twh.size() * sizeof(cpx)));
    CK(cudaMemcpy(tw, twh.data(), twh.size() * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(P, ph.data(), Q * Q * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(da, h.data(), total * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db, h.data(), total * sizeof(cpx), cudaMemcpyHostToDevice));
    using Pc = PipeCfg<N>;
    CK(cudaFuncSetAttribute(k_dbg<N, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Pc::SMEM));
    CK(cudaFuncSetAttribute(k_dbg<N, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Pc::SMEM));
    SweepGeom g{N, Band<N>::lo_end, Band<N>::hi_start, tw};
    const int tiles_x = band_cols(g) / Pc::CW, ntiles = tiles_x * batch;
    CUtensorMap ma, mb;
    tile_map(&ma, da, N, batch, Pc::CW, Pc::BR); tile_map(&mb, db, N, batch, Pc::CW, Pc::BR);
    int nsm = 0; CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, 0));
    const int grid = ntiles < nsm ? ntiles : nsm;
    auto reg = [&] { k_dbg<N, 0><<<grid, Pc::THREADS, Pc::SMEM>>>(ma, P, g.lo_end, g.hi_start, tiles_x, ntiles, tw, nullptr); };
    auto shd = [&] { k_dbg<N, 4><<<grid, Pc::THREADS, Pc::SMEM>>>(mb, P, g.lo_end, g.hi_start, tiles_x, ntiles, tw, nullptr); };
    reg(); shd();
    CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
    std::vector<cpx> a(total), b(total);
    CK(cudaMemcpy(a.data(), da, total * sizeof(cpx), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b.data(), db, total * sizeof(cpx), cudaMemcpyDeviceToHost));
    size_t diff = 0, changed = 0;
    for (size_t i = 0; i < total; i++) { diff += memcmp(&a[i], &b[i], sizeof(cpx)) != 0; changed += memcmp(&a[i], &h[i], sizeof(cpx)) != 0; }
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    std::vector<float> t_reg, t_shd;
    for (int r = 0; r < rounds; r++) {
        for (int v = 0; v < 2; v++) {
            cudaEventRecord(e0);
            for (int k = 0; k < reps; k++) { if (v == 0) reg(); else shd(); }
            cudaEventRecord(e1); cudaEventSynchronize(e1);
            float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
            (v == 0 ? t_reg : t_shd).push_back(ms / reps * 1e3f);
        }
    }
    CK(cudaGetLastError());
    cudaFuncAttributes f0, f1;
    cudaFuncGetAttributes(&f0, k_dbg<N, 0>); cudaFuncGetAttributes(&f1, k_dbg<N, 4>);
    auto stats = [](std::vector<float> v) { std::sort(v.begin(), v.end()); return std::array<float, 3>{v.front(), v[v.size() / 2], v.back()}; };
    const auto sr = stats(t_reg), ss = stats(t_shd);
    printf("N=%4d batch=%2d S6 twiddles A/B, %d rounds x %d launches, us min/median/max | shared (regs=%3d): %.2f / %.2f / %.2f | "
           "registers (regs=%3d): %.2f / %.2f / %.2f | median gain %.1f %% | differing=%zu changed=%zu of %zu\n",
           N, batch, rounds, reps, f1.numRegs, ss[0], ss[1], ss[2], f0.numRegs, sr[0], sr[1], sr[2], 100.0 * (1.0 - sr[1] / ss[1]),
           diff, changed, total);
    cudaFree(da); cudaFree(db); cudaFree(P); cudaFree(tw);
}

int main(int argc, char** argv)
{
    const int reps = 20;
    run_tw_ab<1024>(40, 50, 7);
    run<1024>(8, reps);
    run<1024>(16, reps);
    run<2048>(8, reps);
    run<4096>(2, reps);
    run<512>(32, reps);
    run_dbg<1024, 0>(8, reps); run_dbg<1024, 1>(8, reps); run_dbg<1024, 2>(8, reps); run_dbg<1024, 3>(8, reps);
    run_dbg<2048, 0>(8, reps); run_dbg<2048, 1>(8, reps); run_dbg<2048, 2>(8, reps); run_dbg<2048, 3>(8, reps);
    run_dbg<4096, 0>(2, reps); run_dbg<4096, 1>(2, reps); run_dbg<4096, 2>(2, reps); run_dbg<4096, 3>(2, reps);
    return 0;
}
