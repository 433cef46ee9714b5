// fdes_b200 -- multislice engine: the B200-native replacement for everything below
// buildMeasurements (reference src/crystalMaker.cu:227-424).
#pragma once
#include "kernels.cuh"
#include "params.h"
#include <cuda_runtime.h>
#include <string>
#include <vector>

namespace fdes {

struct EngineOptions {
    int gpu_index = 0;
    int batch = 0;              // phonon configurations advanced together (0 = automatic)
    int rank = 0, world = 1;    // shard of the frozen-phonon configurations handled here
    bool want_exitwave = false; // keep the coherent exit-wave average (print_level 2)
    bool use_graph = true;      // replay the slice loop as a CUDA graph
};

struct EngineTimings {
    double slice_loop_ms = 0.0;     // CUDA-event time spent in the S1..S6 loops
    double atoms_ms = 0.0;          // jitter + binning + sort + row pointers
    long long slices_executed = 0;  // (#sub-slices) x (#configurations) processed by this rank
    long long kernel_launches = 0;  // kernels of this library launched by the engine's calls (graph nodes at every replay)
};

// One simulation = one Params + one atom list on one GPU.
class Engine {
public:
    Engine(const Params& p, const Atoms& atoms, const EngineOptions& opt);
    ~Engine();
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;

    const Params& params() const { return p_; }           // after sub-slicing
    int grid() const { return N_; }
    int num_species() const { return nZ_; }
    int configs_total() const { return count_; }
    int config_begin() const { return j0_; }
    int config_end() const { return j1_; }

    // Partial sums of this rank for measurement index k (tilt/defocus):
    //   intensity_dev()  [m2*m1] float   sum_j |...|^2 / count      (before the detector tail)
    //   exitwave_dev()   [m2*m1] complex sum_j psi_j / count        (only with want_exitwave)
    // External accumulators (e.g. torch tensors that are all-reduced over NCCL) can be
    // installed with set_accumulators before run_k.
    void set_accumulators(float* intensity_dev, cpx* exitwave_dev);
    void run_k(int k);
    float* intensity_dev() { return I_; }
    cpx* exitwave_dev() { return ew_; }
    // adds the partial sums of other engines of this process (possibly on other GPUs: read through
    // NVLink peer mappings, fixed order) to this engine's accumulators; call after every engine's run_k
    void reduce_from(const std::vector<Engine*>& others);
    int gpu_index() const { return opt_.gpu_index; }
    // detector tail of the reference (addNoiseAndMtf + copyMiddleOut) on the (reduced) intensity:
    // image_host [n2*n1]; exitwave_host [m2*m1*2] may be null.
    void finish_k(int k, float* image_host, float* exitwave_host);
    // untilted, phonon-free potential slices with the ORIGINAL slicing (print_level >= 1):
    // out_host [m3_orig][m2][m1][2]
    void potential_slices(float* out_host);

    // --- building blocks exposed for parity tests / benchmarks (device pointers) -------------
    // jittered coordinates of the next configuration -> host (advances the RNG like run_k would)
    void next_jittered_coords(int k, float* xyz_host);
    // integer bin tuples (i1,i2,i3,zidx | -1) for host coordinates [nAt][3]
    void bin_tuples(const float* xyz_host, int* bins_host);
    // phase grating V of slice s for host coordinates -> V_host [m2*m1*2]
    void phase_grating(const float* xyz_host, int s, float* V_host);
    // one multislice run with given coordinates, plane wave / probe of index k; returns the
    // exit wave (real space) in psi_host [m2*m1*2]; trace buffers may be null
    void exit_wave(const float* xyz_host, int k, float* psi_host);
    // throughput loop used by bench.py: `configs` configurations (coordinates resident in HBM,
    // jitter applied if frPh > 0), returns CUDA-event milliseconds of the whole loop
    double bench_configs(int k, int configs);
    // STEM scan: detector sums out_host [nprobes][ndet] for probe positions xy_host [nprobes][2]
    // (metres, relative to the grid centre) and annular detectors det_mrad_host [ndet][2]
    // (inner, outer half-angle in mrad); averaged over this rank's frozen-phonon configurations
    // with weight 1/count.  loop_ms (may be null): CUDA-event time of the scan.
    void stem_scan(int k, int nprobes, const float* xy_host, int ndet, const float* det_mrad_host,
                   float* out_host, double* loop_ms);
    // 4D-STEM scan: out_pattern_host [nprobes][Q/bin][Q/bin] = the diffraction intensity of every probe, fftshifted,
    // cropped to the centred window Q = stem4d_window(N, window, bin) and binned bin x bin, averaged like stem_scan;
    // with ndet > 0 also the annular signals out_det_host [nprobes][ndet], bitwise those of stem_scan.  The raster
    // runs in passes of probes_per_pass probes (0: stem_4d_probes_per_pass), the copy of a finished pass to the
    // host overlapping the next pass.  loop_ms: CUDA-event time of the device loop.
    void stem_scan_4d(int k, int nprobes, const float* xy_host, int window, int bin, int ndet, const float* det_mrad_host,
                      int probes_per_pass, float* out_pattern_host, float* out_det_host, double* loop_ms);
    // automatic pass size: the two device pass buffers take at most about a quarter of the free device memory,
    // and never more than the whole raster
    int stem_4d_probes_per_pass(int nprobes, int window, int bin);
    // average launch duration [ms] of each of the six sweeps on a prepared batch of nb configs
    void time_sweeps(int k, int nb, int reps, float* ms6);
    int batch() const { return B_; }
    int band_columns() const { return g_.lo_end >= g_.hi_start ? N_ : g_.lo_end + (N_ - g_.hi_start); }

    const EngineTimings& timings() const { return tm_; }
    void reset_timings() { tm_ = EngineTimings(); }
    cudaStream_t stream() const { return st_; }

private:
    struct Call;                                    // scope of a public entry point (engine.cu)
    void init(const Atoms& atoms);                  // constructor body (device already selected)
    void release();                                 // stream, events, arena, graph
    void setup_tables();
    void make_incident(int k);                      // psi_in_ (row space) for index k
    // jitter + bin + sort + rowptr of a batch into record set `set` (-1: the active one) on stream st (null: st_)
    void prepare_batch(int nb, const float* xyz_k, int set = -1, cudaStream_t st = nullptr);
    void bin_and_sort(int b0, int nconf, const float* xyz_dev, int set = -1, cudaStream_t st = nullptr);
    void run_batches(int k, int jb, int je, bool reference_order);   // batches of configurations, preparation overlapped
    void slice_loop(int nb);                        // S1..S6 for all slices, batch nb
    void run_slices_plain(int nb);
    void accumulate_outputs(int k, int nb);
    void tilt(float* xyz_dev, float t0, float t1, float t2);
    void specimen_k(int k);                         // xyzK_ <- the specimen of measurement k (offset and tilt)
    // S1 + S2 (W_ <- potentials) and S1..S4 (D <- transmission functions) of a slice pair, from the active record set
    void potential_pair(int s, int s2, int images, int cfg_stride = 1, int cfg_off2 = 0);
    void transmission_pair(int s, int npair, int nb, cpx* D);
    void potential_to_host(int s, float* V_host);   // real-space potential of slice s, absorptive factor applied
    // pieces of the STEM scans (engine.cu)
    DetectorRings stem_rings(int k, int nprobes, int ndet, const float* det_mrad_host, int min_det) const;
    void stem_prepare(int k, int nprobes, const float* xy_host, float* shifts, float* det_out, size_t det_elems);
    void stem_transmission(int k, int j, cpx* tstack);
    void stem_probes(const float* shifts, int nb, const cpx* tstack);

    Params p_;
    EngineOptions opt_;
    int N_ = 0, nZ_ = 0, nAt_ = 0, count_ = 1, j0_ = 0, j1_ = 1, B_ = 1;
    int m3_orig_ = 1; float d3_orig_ = 0.f;
    std::vector<int> Zlist_;
    SweepGeom g_{};
    cudaStream_t st_ = nullptr, st_prep_ = nullptr;     // sweeps; atom preparation of the next batch
    cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
    cudaEvent_t ev_ready_ = nullptr, ev_prep_[2] = {nullptr, nullptr}, ev_used_[2] = {nullptr, nullptr};
    // per-batch atom records (deposit records sorted by (slice, species, row), row pointers, jittered coordinates)
    struct RecordSet {
        uint32_t* keys = nullptr;
        int *cols = nullptr, *rowptr = nullptr;
        float *w = nullptr, *xyzFP = nullptr;
    };
    RecordSet rs_[2];
    int act_ = 0;               // record set the sweeps read
    // device memory
    cpx *tw_ = nullptr, *Pq_ = nullptr, *psi_in_ = nullptr, *Psi_ = nullptr, *W_ = nullptr, *D_ = nullptr, *A_ = nullptr;
    cpx *ew_ = nullptr, *ew_own_ = nullptr, *lens_ = nullptr, *scratch_ = nullptr;
    float *Gq_ = nullptr, *I_ = nullptr, *I_own_ = nullptr, *det_ = nullptr, *J_ = nullptr;
    float *xyz0_ = nullptr, *xyzTO_ = nullptr, *xyzK_ = nullptr, *dwf_ = nullptr, *occ_ = nullptr;
    int* zidx_ = nullptr;
    void* rng_ = nullptr;
    unsigned char* rng_bytes_ = nullptr;
    unsigned char* noise_rng_ = nullptr;   // per-pixel XORWOW states of the Poisson noise (pixel_dose > 0)
    void* arena_ = nullptr;           // the one device block all buffers above are carved from
    std::vector<cpx> tw_host_;
    long long rng_pos_ = 0;     // normals every XORWOW stream has produced so far
    long long rng_target_ = 0;  // position of the next configuration in the reference's (k, j) order
    uint32_t* keys_tmp_ = nullptr;
    int *cols_tmp_ = nullptr, *bins_ = nullptr;
    float* w_tmp_ = nullptr;
    unsigned int* hist_ = nullptr;
    double *norm_partial_ = nullptr, *norm_result_ = nullptr;
    size_t rec_stride_ = 0, rp_stride_ = 0;
    bool fuse_ctf_ = false;           // imaging mode on pipelined column kernels: the CTF rides on the last slice's S6 (when no exit wave is kept)
    void ensure_lens(int k);
    bool plane_first_slice_ = false;  // plane-wave illumination on pipelined column kernels: slice 0 runs S6 from D, no S5
    int mask_E_ = 0;                  // points per thread of a line (row-mask layout); 0: no masks
    int nkeys_ = 0, key_bits_ = 0, nrec_ = 0;
    int lens_k_ = -1, incident_k_ = -1;
    cudaGraphExec_t graph_[2] = {nullptr, nullptr};     // slice loop of a batch, per record set
    int graph_nb_[2] = {0, 0};
    long long graph_launches_[2] = {0, 0};              // kernels of each graph
    bool warmed_ = false;
    EngineTimings tm_;
    bool in_call_ = false;            // inside a public entry point (Call)
};

// frees the device blocks cached between simulations (idle ones)
void release_device_cache();

// Side Q of the 4D-STEM window on an N x N grid (host only; throws with the reason when not admissible):
// window > 0 is taken as is when 1 <= window <= N, window = N (mod 2) and bin divides it; window = 0 is the smallest
// such Q that holds every frequency the 2/3 band limit keeps.
int stem4d_window(int N, int window, int bin);

}  // namespace fdes
