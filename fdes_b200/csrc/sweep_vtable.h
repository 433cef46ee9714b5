// fdes_b200 -- run-time dispatch over the grid sizes the fast sweeps are instantiated for.
// Every size lives in its own translation unit (sweeps_size.cu compiled with -DFDES_SWEEP_N=<N>),
// so the sizes build in parallel; sweeps.cu selects the table of launchers by N.
#pragma once
#include "kernels.cuh"
#include <vector>

// grid sizes with register-resident Stockham line transforms (E points per thread, see
// fft_core.cuh): powers of two and the 2^a 5^b sizes of the reference's shipped examples
#define FDES_SWEEP_SIZES(X) X(64) X(128) X(256) X(512) X(1024) X(2048) X(4096) X(320) X(800) X(1000)

struct CUtensorMap_st;   // <cuda.h>

namespace fdes {

// TMA descriptor (cached per device / array / geometry) of an [nimg][N][N] complex64 array with
// boxes of [BR rows][CW columns] -- the column tiles of col_pipe.cuh (tma_map.cu)
void tile_map(CUtensorMap_st* out, const void* base, int N, int nimg, int CW, int BR);

struct SweepVTable {
    int N, rows_per_block, cols_per_block, line_points;
    void (*density_rows)(const SweepGeom&, cpx*, const int*, const int*, const float*, int, int, int, int, size_t, size_t, int, int, cudaStream_t);
    void (*potential_cols)(const SweepGeom&, cpx*, const cpx*, const float*, const int*, int, int, int, int, size_t, int, int, cudaStream_t);
    void (*transmit_rows)(const SweepGeom&, const cpx*, cpx*, int, float, int, cudaStream_t);
    void (*bandlimit_cols)(const SweepGeom&, cpx*, int, int, cudaStream_t);
    void (*multiply_rows)(const SweepGeom&, cpx*, const cpx*, size_t, int, bool, cudaStream_t);
    void (*propagate_cols)(const SweepGeom&, cpx*, const cpx*, int, cudaStream_t);
    void (*rows_fft)(const SweepGeom&, const void*, void*, int, RowEpilogue, const RowOpts&, int, cudaStream_t);
    void (*rows_fft_sum)(const SweepGeom&, const cpx*, void*, int, RowEpilogue, const RowOpts&, int, cudaStream_t);
    void (*cols_fft)(const SweepGeom&, const cpx*, void*, int, ColOp, const void*, float, int, cudaStream_t);
    void (*probe_cols)(const SweepGeom&, cpx*, const cpx*, const float*, int, cudaStream_t);
    int (*detector_tiles)(const SweepGeom&);
    void (*detector_cols)(const SweepGeom&, const cpx*, float*, float*, const DetectorRings&, float, float, float, int, cudaStream_t);
    void (*detector4d_cols)(const SweepGeom&, const cpx*, float*, float*, int, int, float, int, cudaStream_t);
    std::vector<cpx> (*make_twiddles)(int N);
    // null where pipelined is false: S6 reading another image stack, see launch_propagate_cols_from
    void (*propagate_cols_from)(const SweepGeom&, cpx*, const cpx*, int, int, const cpx*, int, bool, const cpx*, cudaStream_t);
    bool pipelined;           // the column sweeps of this size run on the TMA pipeline
};

// any other even size: mixed-radix line transforms in shared memory with run-time N (generic_sweeps.cu)
bool generic_size_supported(int N);
const SweepVTable* generic_sweep_vtable();
// true when N runs on the register-resident kernels (band-limited column range, pair packing ...)
bool fft_size_is_fast(int N);

// one per size, defined in that size's translation unit
#define FDES_DECLARE_VT(N_) const SweepVTable* sweep_vtable_##N_();
FDES_SWEEP_SIZES(FDES_DECLARE_VT)
#undef FDES_DECLARE_VT

}  // namespace fdes
