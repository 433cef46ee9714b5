// fdes_b200 -- run-time dispatch of the multislice sweeps (kernels: sweep_kernels.cuh, one
// translation unit per grid size: sweeps_size.cu).  Replaces the cuFFT + cuBLAS +
// one-thread-per-pixel chain of the reference's per-slice loop (phaseGrating,
// src/crystalMaker.cu:507-536; forwardPropagation, src/multisliceSimulation.cu:538-611).
#include "sweep_vtable.h"
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>

namespace fdes {

// read by pipe_grid (sweep_kernels.cuh), which every size's translation unit compiles
thread_local int pipe_cta_cap = 0;
thread_local int pipe_last_grid = 0;
thread_local long long launch_tally = 0;

// Function attributes are per device: the dynamic shared-memory limit is raised per kernel and device, and only
// when a launch needs more than was set before, so launches into a stream capture do not touch the attribute.
static void allow_smem(const void* kernel, size_t bytes)
{
    if (bytes <= 48 * 1024) return;
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> have;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    size_t& cur = have[{kernel, dev}];
    if (bytes > cur) {
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
}

void launch_args(const void* kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, void** args)
{
    allow_smem(kernel, smem);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelExC(&cfg, kernel, args);
    if (e != cudaSuccess) {
        cudaGetLastError();     // reported here; not again by a later check
        const char* name = nullptr;
        if (cudaFuncGetName(&name, kernel) != cudaSuccess || !name) name = "?";
        throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " launching " + name);
    }
    launch_tally++;
}

static const SweepVTable* find_fast_vtable(int N)
{
    switch (N) {
#define FDES_VT_CASE(N_) case N_: return sweep_vtable_##N_();
        FDES_SWEEP_SIZES(FDES_VT_CASE)
#undef FDES_VT_CASE
        default: return nullptr;
    }
}
static const SweepVTable* find_vtable(int N)
{
    if (const SweepVTable* t = find_fast_vtable(N)) return t;
    return generic_size_supported(N) ? generic_sweep_vtable() : nullptr;
}
static const SweepVTable& vt(int N)
{
    const SweepVTable* t = find_vtable(N);
    if (!t) throw std::runtime_error("grid size " + std::to_string(N) + " unsupported: sample size (image + 2*border) must be 8 .. 8192");
    return *t;
}

bool fft_size_supported(int N) { return find_vtable(N) != nullptr; }
bool fft_size_is_fast(int N) { return find_fast_vtable(N) != nullptr; }
std::vector<cpx> make_twiddles(int N) { return vt(N).make_twiddles(N); }
SweepGeom make_sweep_geom(int N, const cpx* tw, int mask_off)
{
    vt(N);
    SweepGeom g{N, N, N, tw, mask_off};
    // the generic sweeps transform every column (the band limit is applied by the mask alone)
    if (!fft_size_is_fast(N)) return g;
    // 2/3 band limit: largest |i1| kept on the axis by zeroHighFreq's float test, bounds rounded outwards
    // to multiples of 32; no column skipped when the two ranges meet
    int kb = 0;
    const float mind = (float)N;
    while (kb + 1 <= N / 2 && !(((float)((kb + 1) * (kb + 1)) * 9.f / (mind * mind)) > 1.f)) kb++;
    const int lo_end = ((kb + 1 + 31) / 32) * 32, hi_start = ((N - kb) / 32) * 32;
    if (lo_end < hi_start) { g.lo_end = lo_end; g.hi_start = hi_start; }
    return g;
}
int rows_per_block(int N) { return vt(N).rows_per_block; }
int cols_per_block(int N) { return vt(N).cols_per_block; }
int line_points(int N) { return vt(N).line_points; }
bool sweeps_pipelined(int N) { return vt(N).pipelined; }

void launch_density_rows(const SweepGeom& g, cpx* A, const int* rowptr, const int* rec_col, const float* rec_w,
                         int slice, int slice2, int nZ, int batch, size_t rec_stride, size_t rowptr_stride, cudaStream_t st,
                         int cfg_stride, int cfg_off2)
{
    vt(g.N).density_rows(g, A, rowptr, rec_col, rec_w, slice, slice2, nZ, batch, rec_stride, rowptr_stride, cfg_stride, cfg_off2, st);
}
void launch_potential_cols(const SweepGeom& g, cpx* B, const cpx* A, const float* Gq, const int* rowptr, int slice,
                           int slice2, int nZ, int batch, size_t rowptr_stride, cudaStream_t st, int cfg_stride, int cfg_off2)
{
    vt(g.N).potential_cols(g, B, A, Gq, rowptr, slice, slice2, nZ, batch, rowptr_stride, cfg_stride, cfg_off2, st);
}
void launch_transmit_rows(const SweepGeom& g, const cpx* W, cpx* D, int npair, float imPot, int batch, cudaStream_t st)
{
    vt(g.N).transmit_rows(g, W, D, npair, imPot, batch, st);
}
void launch_bandlimit_cols(const SweepGeom& g, cpx* W, int batch, int npair, cudaStream_t st)
{
    vt(g.N).bandlimit_cols(g, W, batch, npair, st);
}
void launch_multiply_rows(const SweepGeom& g, cpx* Psi, const cpx* E, size_t e_batch_stride, int batch, bool psi_full,
                          cudaStream_t st)
{
    vt(g.N).multiply_rows(g, Psi, E, e_batch_stride, batch, psi_full, st);
}
void launch_propagate_cols(const SweepGeom& g, cpx* Psi, const cpx* Pq, int batch, cudaStream_t st)
{
    vt(g.N).propagate_cols(g, Psi, Pq, batch, st);
}
void launch_propagate_cols_from(const SweepGeom& g, cpx* out, const cpx* src, int src_img_stride, int src_images, const cpx* Pq,
                                int batch, bool times_n, const cpx* lens, cudaStream_t st)
{
    const SweepVTable& t = vt(g.N);
    if (!t.propagate_cols_from)
        throw std::runtime_error("grid size " + std::to_string(g.N) + ": S6 from another image stack needs the pipelined column sweeps");
    t.propagate_cols_from(g, out, src, src_img_stride, src_images, Pq, batch, times_n, lens, st);
}
void launch_rows_fft(const SweepGeom& g, const void* in, void* out, int dir, RowEpilogue epi, const RowOpts& o, int batch,
                     cudaStream_t st)
{
    vt(g.N).rows_fft(g, in, out, dir, epi, o, batch, st);
}
void launch_rows_fft_sum(const SweepGeom& g, const cpx* in, void* out, int dir, RowEpilogue epi, const RowOpts& o, int nb,
                         cudaStream_t st)
{
    vt(g.N).rows_fft_sum(g, in, out, dir, epi, o, nb, st);
}
void launch_cols_fft(const SweepGeom& g, const cpx* in, void* out, int dir, ColOp op, const void* table, float scale,
                     int batch, cudaStream_t st)
{
    vt(g.N).cols_fft(g, in, out, dir, op, table, scale, batch, st);
}
void launch_probe_cols(const SweepGeom& g, cpx* Psi, const cpx* PSI0, const float* shifts, int batch, cudaStream_t st)
{
    vt(g.N).probe_cols(g, Psi, PSI0, shifts, batch, st);
}
int detector_tiles(const SweepGeom& g) { return vt(g.N).detector_tiles(g); }
void launch_detector_cols(const SweepGeom& g, const cpx* Psi, float* partial, float* out, const DetectorRings& rings,
                          float d1, float d2, float weight, int batch, cudaStream_t st)
{
    vt(g.N).detector_cols(g, Psi, partial, out, rings, d1, d2, weight, batch, st);
}
void launch_detector4d_cols(const SweepGeom& g, const cpx* Psi, float* scratch, float* out, int Q, int bin, float weight,
                            int batch, cudaStream_t st)
{
    if (Q < 1 || Q > g.N || (Q - g.N) % 2 != 0 || bin < 1 || Q % bin != 0)
        throw std::runtime_error("4D-STEM window " + std::to_string(Q) + " / bin " + std::to_string(bin) + " not admissible at N = " +
                                 std::to_string(g.N));
    vt(g.N).detector4d_cols(g, Psi, scratch, out, Q, bin, weight, batch, st);
}

}  // namespace fdes
