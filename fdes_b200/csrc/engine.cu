// fdes_b200 -- multislice engine (host orchestration of the sm_100a sweeps).
// Mirrors the k / j / s loop structure of buildMeasurements (reference
// src/crystalMaker.cu:227-424) with a different execution plan:
//   * all per-simulation constants (propagator, scattering factors, twiddles, lens and detector
//     tables) are computed once instead of once per slice;
//   * atoms are binned and sorted once per phonon configuration instead of being scanned
//     m3*nZ times;
//   * B phonon configurations advance together through the six sweeps of a slice;
//   * the wave function stays in the row-transformed (kx, y) domain between slices.
#include "engine.h"
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <mutex>
#include <stdexcept>
#include <vector>

namespace fdes {

namespace {
struct PhaseTimer {
    bool on = getenv("FDES_B200_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void mark(const char* what)
    {
        if (!on) return;
        const auto n = std::chrono::steady_clock::now();
        fprintf(stderr, "    [engine] %-22s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};
}  // namespace

// Every public entry point runs on the engine's own device, whatever the caller's current device
// is (torch switching devices, several engines of one process on different GPUs), and restores
// the caller's device on the way out (Engine::Call).
namespace {
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) {
            cudaError_t e_ = cudaSetDevice(dev);
            if (e_ != cudaSuccess)
                throw std::runtime_error(std::string("cudaSetDevice(") + std::to_string(dev) + "): " + cudaGetErrorString(e_));
            changed = true;
        }
    }
    ~DeviceGuard() { if (changed && prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
}  // namespace

// The scope of a public entry point: the engine's device, and the kernels the call launched (the growth of
// launch_tally) added to EngineTimings::kernel_launches.  A call made from inside another one
// (stem_scan_4d -> stem_4d_probes_per_pass) is counted by the outer call.
struct Engine::Call {
    Engine& e;
    DeviceGuard device;
    const bool outer;
    const long long tally0;
    explicit Call(Engine& eng) : e(eng), device(eng.opt_.gpu_index), outer(!eng.in_call_), tally0(launch_tally) { e.in_call_ = true; }
    ~Call()
    {
        if (!outer) return;
        e.tm_.kernel_launches += launch_tally - tally0;
        e.in_call_ = false;
    }
    Call(const Call&) = delete;
    Call& operator=(const Call&) = delete;
};

// ---------------------------------------------------------------------------------------------
// Device memory: every buffer of an Engine is a slice of ONE block, and blocks are cached per
// process between simulations (the reference cudaMalloc/cudaFree's its buffers per call and
// even per slice, src/crystalMaker.cu:255-265, 516-535; cudaMalloc/cudaFree of ~30 buffers cost
// tens of milliseconds and a device synchronisation each, which would dominate a drop-in FDES()
// call whose multislice work is a few milliseconds).
// ---------------------------------------------------------------------------------------------
namespace {
struct PoolBlock { void* ptr; size_t bytes; int device; bool in_use; };
std::mutex g_pool_mutex;
std::vector<PoolBlock> g_pool;
constexpr size_t kPoolKeepBytes = (size_t)8 << 30;   // free cached blocks beyond this total

void* pool_acquire(size_t bytes, int device)
{
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    int best = -1;
    for (int i = 0; i < (int)g_pool.size(); i++) {
        const PoolBlock& b = g_pool[i];
        if (!b.in_use && b.device == device && b.bytes >= bytes && (best < 0 || b.bytes < g_pool[best].bytes)) best = i;
    }
    if (best >= 0 && g_pool[best].bytes <= 2 * bytes + ((size_t)64 << 20)) {
        g_pool[best].in_use = true;
        return g_pool[best].ptr;
    }
    const size_t granule = (size_t)32 << 20;
    const size_t want = (bytes + granule - 1) / granule * granule;
    void* p = nullptr;
    cudaError_t err = cudaMalloc(&p, want);
    if (err != cudaSuccess) {
        // drop every cached free block of this device and retry once
        for (auto it = g_pool.begin(); it != g_pool.end();) {
            if (!it->in_use && it->device == device) { cudaFree(it->ptr); it = g_pool.erase(it); }
            else ++it;
        }
        cudaGetLastError();
        err = cudaMalloc(&p, want);
    }
    if (err != cudaSuccess)
        throw std::runtime_error(std::string("cudaMalloc of ") + std::to_string(want >> 20) + " MiB failed: " + cudaGetErrorString(err));
    g_pool.push_back({p, want, device, true});
    return p;
}
void pool_release(void* ptr)
{
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    size_t free_bytes = 0;
    for (PoolBlock& b : g_pool) {
        if (b.ptr == ptr) b.in_use = false;
        if (!b.in_use) free_bytes += b.bytes;
    }
    // keep the cache bounded: free the largest idle blocks first
    while (free_bytes > kPoolKeepBytes) {
        int big = -1;
        for (int i = 0; i < (int)g_pool.size(); i++)
            if (!g_pool[i].in_use && (big < 0 || g_pool[i].bytes > g_pool[big].bytes)) big = i;
        if (big < 0) break;
        cudaFree(g_pool[big].ptr);
        free_bytes -= g_pool[big].bytes;
        g_pool.erase(g_pool.begin() + big);
    }
}
// buffers are registered first, then carved out of one block
struct ArenaPlan {
    std::vector<std::pair<void**, size_t>> reqs;
    template <typename T>
    void add(T*& p, size_t n) { reqs.push_back({reinterpret_cast<void**>(&p), std::max<size_t>(n, 1) * sizeof(T)}); }
    static size_t align(size_t b) { return (b + 255) & ~(size_t)255; }
    size_t total() const { size_t t = 0; for (auto& r : reqs) t += align(r.second); return t; }
    void assign(void* base) const
    {
        char* q = static_cast<char*>(base);
        for (auto& r : reqs) { *r.first = q; q += align(r.second); }
    }
};
}  // namespace

void release_device_cache()
{
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    for (auto it = g_pool.begin(); it != g_pool.end();) {
        if (!it->in_use) { cudaFree(it->ptr); it = g_pool.erase(it); }
        else ++it;
    }
}

Engine::Engine(const Params& pin, const Atoms& atoms, const EngineOptions& opt) : p_(pin), opt_(opt)
{
    if (atoms.size() <= 0) throw std::runtime_error("no atoms in the specimen");
    if (p_.mode < 0 || p_.mode > 2) throw std::runtime_error("mode must be 0 (imaging), 1 (DP) or 2 (CBED)");
    if (p_.m1 != p_.m2)
        throw std::runtime_error("non-square grids are not supported (the reference's phaseGrating "
                                 "uses a transposed cuFFT plan for m1 != m2, src/crystalMaker.cu:575)");
    if (!fft_size_supported(p_.m1))
        throw std::runtime_error("grid size " + std::to_string(p_.m1) +
                                 " unsupported: sample size (image + 2*border) must be between 8 and 8192");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw std::runtime_error("no CUDA device: fdes_b200 has no CPU fallback");
    if (opt_.gpu_index < 0 || opt_.gpu_index >= ndev)
        throw std::runtime_error("gpu index " + std::to_string(opt_.gpu_index) + " out of range (" + std::to_string(ndev) + " device(s))");
    const Call call(*this);
    try {
        init(atoms);
    } catch (...) {
        release();     // the destructor does not run for a throwing constructor
        throw;
    }
}

void Engine::init(const Atoms& atoms)
{
    PhaseTimer pt;

    // sub-slicing (subSliceRatio / setSubSlices, src/crystalMaker.cu:246-247, 720-743)
    m3_orig_ = p_.m3; d3_orig_ = p_.d3;
    const float ratio = sub_slice_ratio(p_.d3, p_.subSlTh);
    set_sub_slices(p_, ratio);
    if (p_.m3 < 1) throw std::runtime_error("sample_size_z must be >= 1");

    N_ = p_.m1;
    nAt_ = atoms.size();
    p_.nAt = nAt_;
    Zlist_ = list_of_elements(atoms.Z);
    nZ_ = (int)Zlist_.size();
    count_ = p_.frPh > 0 ? p_.frPh : 1;
    const int world = std::max(1, opt_.world), rank = std::min(std::max(0, opt_.rank), world - 1);
    j0_ = (int)(((long long)count_ * rank) / world);
    j1_ = (int)(((long long)count_ * (rank + 1)) / world);
    const int mine = std::max(1, j1_ - j0_);
    // configurations advanced together: about 80 Mpixel per launch, at least 10 and at most 40 configurations
    // (40 at 1024^2 and below, 20 at 2048^2, 10 at 4096^2).  Every sweep is one launch over the batch; the
    // longer the launch, the less its ramp-up and tail weigh (measured, same box: 1024^2 55.5 / 59.0 / 60.6 /
    // 61.7 Gpx*slices/s at 10 / 20 / 30 / 40; 2048^2 53.3 / 54.3 / 54.7 / 54.7 at 10 / 16 / 20 / 26; 4096^2
    // 29.9 / 28.4 at 10 / 16), and the batch buffers ((4 + nZ) complex grids per configuration) stay far below
    // the 180 GB of HBM
    const long long fit = (80LL << 20) / ((long long)N_ * N_);
    B_ = opt_.batch > 0 ? opt_.batch : (int)std::min(40LL, std::max(10LL, fit));
    while (B_ > 1 && (size_t)B_ * (4 + nZ_) * (size_t)N_ * N_ * sizeof(cpx) > ((size_t)48 << 30)) B_ /= 2;
    if (opt_.batch <= 0) B_ = std::min(B_, mine);   // an explicit batch is honoured (STEM probes batch independently of the phonon count)
    const long long nk = (long long)p_.m3 * nZ_ * N_;
    if (nk >= (1LL << 31) - 2) throw std::runtime_error("slices * species * rows too large for 32-bit row keys");
    nkeys_ = (int)nk;
    key_bits_ = 0;
    while ((1LL << key_bits_) <= nk) key_bits_++;
    nrec_ = 4 * nAt_;
    rec_stride_ = (size_t)nrec_;
    // row pointers of a configuration, followed by its row masks (launch_row_masks)
    mask_E_ = line_points(N_);
    rp_stride_ = (size_t)nkeys_ + 1 + (mask_E_ > 0 ? (size_t)(nkeys_ / N_) * (N_ / mask_E_) : 0);

    pt.mark("ctor: host prep");
    CK(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&st_prep_, cudaStreamNonBlocking));
    CK(cudaEventCreate(&ev0_));
    CK(cudaEventCreate(&ev1_));
    CK(cudaEventCreateWithFlags(&ev_ready_, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
        CK(cudaEventCreateWithFlags(&ev_prep_[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_used_[i], cudaEventDisableTiming));
    }

    const size_t NN = (size_t)N_ * N_, Q = (size_t)(N_ / 2 + 1);
    tw_host_ = make_twiddles(N_);
    ArenaPlan plan;
    plan.add(tw_, tw_host_.size());
    plan.add(Pq_, Q * Q); plan.add(Gq_, (size_t)nZ_ * Q * Q);
    plan.add(psi_in_, NN); plan.add(Psi_, (size_t)B_ * NN); plan.add(W_, (size_t)B_ * NN); plan.add(D_, 2 * (size_t)B_ * NN);
    plan.add(A_, (size_t)B_ * nZ_ * NN);
    plan.add(I_own_, NN); plan.add(lens_, NN); plan.add(det_, NN); plan.add(scratch_, NN);
    plan.add(J_, (size_t)p_.n1 * p_.n2);
    if (opt_.want_exitwave) plan.add(ew_own_, NN);
    plan.add(xyz0_, 3 * (size_t)nAt_); plan.add(xyzTO_, 3 * (size_t)nAt_); plan.add(xyzK_, 3 * (size_t)nAt_);
    plan.add(dwf_, nAt_); plan.add(occ_, nAt_); plan.add(zidx_, nAt_);
    // two sets of per-batch atom records: the records of batch i+1 are prepared on a second stream
    // while the sweeps of batch i read theirs
    for (RecordSet& r : rs_) {
        plan.add(r.xyzFP, (size_t)B_ * 3 * nAt_);
        plan.add(r.keys, (size_t)B_ * nrec_); plan.add(r.cols, (size_t)B_ * nrec_); plan.add(r.w, (size_t)B_ * nrec_);
        plan.add(r.rowptr, (size_t)B_ * rp_stride_);
    }
    plan.add(keys_tmp_, (size_t)B_ * nrec_); plan.add(cols_tmp_, (size_t)B_ * nrec_); plan.add(w_tmp_, (size_t)B_ * nrec_);
    plan.add(bins_, 4 * (size_t)nAt_);
    plan.add(hist_, (size_t)B_ * 256 * sort_num_blocks(nrec_));
    plan.add(norm_partial_, 256); plan.add(norm_result_, 1);
    if (p_.frPh > 0) plan.add(rng_bytes_, rng_state_bytes() * 3 * (size_t)nAt_);
    if (p_.pD > FLT_EPSILON) plan.add(noise_rng_, rng_state_bytes() * NN);   // one XORWOW stream per pixel
    pt.mark("ctor: stream+twiddles");
    arena_ = pool_acquire(plan.total(), opt_.gpu_index);
    pt.mark("ctor: arena");
    plan.assign(arena_);
    rng_ = rng_bytes_;
    I_ = I_own_; ew_ = ew_own_;
    std::vector<int> zidx(nAt_);
    for (int i = 0; i < nAt_; i++)
        zidx[i] = (int)(std::find(Zlist_.begin(), Zlist_.end(), atoms.Z[i]) - Zlist_.begin());
    CK(cudaMemcpyAsync(zidx_, zidx.data(), nAt_ * sizeof(int), cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(xyz0_, atoms.xyz.data(), 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(dwf_, atoms.dwf.data(), nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(occ_, atoms.occ.data(), nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    CK(cudaStreamSynchronize(st_));   // host vectors above go out of scope
    pt.mark("ctor: uploads");

    // coordinates with the tilt offset (src/crystalMaker.cu:282-283)
    CK(cudaMemcpyAsync(xyzTO_, xyz0_, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st_));
    tilt(xyzTO_, p_.tilt_off[0], p_.tilt_off[1], p_.tilt_off[2]);

    // Poisson-noise streams: seed 1 + n3, one per pixel (src/crystalMaker.cu:295)
    if (p_.pD > FLT_EPSILON) launch_rng_init(noise_rng_, (int)NN, 1ULL + (unsigned long long)p_.n3, st_);
    if (p_.frPh > 0) launch_rng_init(rng_, 3 * nAt_, 1ULL, st_);   // seed 1, src/crystalMaker.cu:292
    setup_tables();
    CK(cudaStreamSynchronize(st_));
    pt.mark("ctor: rng+tables");
}

Engine::~Engine()
{
    try {
        DeviceGuard guard(opt_.gpu_index);
        release();
    } catch (...) {
    }
}

void Engine::release()
{
    for (cudaGraphExec_t& g : graph_) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    if (st_prep_) cudaStreamSynchronize(st_prep_);
    if (st_) cudaStreamSynchronize(st_);
    if (arena_) { pool_release(arena_); arena_ = nullptr; }
    if (ev0_) { cudaEventDestroy(ev0_); ev0_ = nullptr; }
    if (ev1_) { cudaEventDestroy(ev1_); ev1_ = nullptr; }
    if (ev_ready_) { cudaEventDestroy(ev_ready_); ev_ready_ = nullptr; }
    for (int i = 0; i < 2; i++) {
        if (ev_prep_[i]) { cudaEventDestroy(ev_prep_[i]); ev_prep_[i] = nullptr; }
        if (ev_used_[i]) { cudaEventDestroy(ev_used_[i]); ev_used_[i] = nullptr; }
    }
    if (st_prep_) { cudaStreamDestroy(st_prep_); st_prep_ = nullptr; }
    if (st_) { cudaStreamDestroy(st_); st_ = nullptr; }
}

void Engine::setup_tables()
{
    // pass twiddle tables (double precision on the host)
    CK(cudaMemcpyAsync(tw_, tw_host_.data(), tw_host_.size() * sizeof(cpx), cudaMemcpyHostToDevice, st_));

    // band columns of the 2/3 limit; the row masks follow the nkeys + 1 row pointers of a configuration
    g_ = make_sweep_geom(N_, tw_, mask_E_ > 0 ? nkeys_ + 1 : 0);
    {
        const char* e = getenv("FDES_B200_NO_FIRST_SLICE_SHORTCUT");     // A/B switch
        plane_first_slice_ = p_.mode != 2 && !p_.doBeamTilt && sweeps_pipelined(N_) && !(e && e[0] == '1');
        fuse_ctf_ = p_.mode == 0 && sweeps_pipelined(N_) && !(e && e[0] == '1');
    }

    launch_propagator_table(Pq_, N_, p_.d1, p_.d2, p_.d3, p_.lambda, p_.cst_pi, st_);
    const size_t Q = (size_t)(N_ / 2 + 1);
    for (int z = 0; z < nZ_; z++)
        launch_scattering_table(Gq_ + (size_t)z * Q * Q, N_, kirkland_row(Zlist_[z]), p_.d1, p_.d2, p_.sigma, p_.cst_pi, st_);
}

void Engine::tilt(float* xyz, float t0, float t1, float t2)
{
    // tiltCoordinates, src/crystalMaker.cu:427-454
    if (fabsf(t2) > FLT_EPSILON) launch_rot(xyz, nAt_, 0, 1, cosf(t2), -sinf(t2), st_);
    if (fabsf(t1) > FLT_EPSILON) launch_rot(xyz, nAt_, 0, 2, cosf(t1), -sinf(t1), st_);
    if (fabsf(t0) > FLT_EPSILON) launch_rot(xyz, nAt_, 1, 2, cosf(t0), -sinf(t0), st_);
}

// the specimen of measurement k in xyzK_: offset and tilt (src/crystalMaker.cu:282-283, 427-454)
void Engine::specimen_k(int k)
{
    CK(cudaMemcpyAsync(xyzK_, xyzTO_, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st_));
    tilt(xyzK_, p_.tiltspec[2 * k], p_.tiltspec[2 * k + 1], 0.f);
}

void Engine::set_accumulators(float* intensity_dev, cpx* exitwave_dev)
{
    I_ = intensity_dev ? intensity_dev : I_own_;
    ew_ = exitwave_dev ? exitwave_dev : ew_own_;
}

static LensParams lens_params(const Params& p, int k, int mode)
{
    LensParams lp;
    for (int a = 0; a < AB_COUNT; a++) { lp.ab0[a] = p.ab0[a]; lp.ab1[a] = p.ab1[a]; }
    lp.defocus_k = p.defoci[k];
    lp.defocspread = p.defocspread; lp.lambda = p.lambda; lp.d1 = p.d1; lp.d2 = p.d2;
    lp.ObjAp = p.ObjAp; lp.pi = p.cst_pi; lp.mode = mode;
    return lp;
}

// incomingWave, src/multisliceSimulation.cu:563-591 -> psi_in_ in the (kx, y) domain
void Engine::make_incident(int k)
{
    if (incident_k_ == k) return;
    const size_t NN = (size_t)N_ * N_;
    RowOpts ro;
    if (p_.mode == 2) {
        // aperture * exp(-i chi) on the Fourier grid, inverse 2-D transform, fftshift
        launch_lens_table(scratch_, N_, lens_params(p_, k, 2), 1.f, st_);
        launch_cols_fft(g_, scratch_, scratch_, +1, COL_PLAIN, nullptr, 1.f, 1, st_);
        launch_rows_fft(g_, scratch_, psi_in_, +1, ROW_STORE_SHIFT, ro, 1, st_);
        // bandwidthLimit (:552-560): FFT2, 2/3 mask, IFFT2, 1/N -- left in row space
        ro.band_only_out = true;
        launch_rows_fft(g_, psi_in_, psi_in_, -1, ROW_STORE, ro, 1, st_);
        launch_bandlimit_cols(g_, psi_in_, 1, 0, st_);
        // normalise to n1*n2 total intensity; psi = IFFT_row(Psi) => sum |psi|^2 = N * sum |Psi|^2
        launch_norm2(psi_in_, NN, norm_partial_, norm_result_, st_);
        double s = 0.0;
        CK(cudaMemcpyAsync(&s, norm_result_, sizeof(double), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        const float nrm = (float)sqrt(s * (double)N_);
        const float alpha = sqrtf((float)(p_.n1 * p_.n2)) / nrm;
        launch_scale_cpx(psi_in_, NN, alpha, st_);
    } else {
        launch_plane_wave_rowspace(psi_in_, N_, 1, st_);
    }
    if (p_.doBeamTilt) {
        // phase ramp in real space (tiltBeam_d, :89-120)
        RowOpts r2;
        r2.band_only_in = (p_.mode == 2);
        launch_rows_fft(g_, psi_in_, scratch_, +1, ROW_STORE, r2, 1, st_);
        launch_tilt_beam(scratch_, N_, p_.d1, p_.d2, p_.lambda, p_.tiltbeam[2 * k], p_.tiltbeam[2 * k + 1],
                         p_.cst_pi, 1, st_);
        RowOpts r3;
        if (p_.mode == 0 || p_.mode == 1) {
            launch_tukey_window(scratch_, N_, p_.dn1, p_.dn2, p_.cst_pi, st_);
            r3.band_only_out = true;
            launch_rows_fft(g_, scratch_, psi_in_, -1, ROW_STORE, r3, 1, st_);
            launch_bandlimit_cols(g_, psi_in_, 1, 0, st_);
        } else {
            r3.scale = 1.f / (float)N_;   // row-space convention: Psi = FFT_row(psi) / N
            launch_rows_fft(g_, scratch_, psi_in_, -1, ROW_STORE, r3, 1, st_);
        }
    }
    incident_k_ = k;
}

// records of `nconf` configurations (slots b0 .. b0+nconf-1) from coordinates [nconf][nAt][3], into
// record set `set` (default: the active one) on stream `st` (default: the engine's)
void Engine::bin_and_sort(int b0, int nconf, const float* xyz_dev, int set, cudaStream_t st)
{
    if (set < 0) set = act_;
    if (!st) st = st_;
    const RecordSet& r = rs_[set];
    BinGeom bg{N_, N_, p_.m3, nZ_, p_.d1, p_.d2, p_.d3};
    SortBuffers sb{r.keys + (size_t)b0 * nrec_, keys_tmp_, r.cols + (size_t)b0 * nrec_, cols_tmp_,
                   r.w + (size_t)b0 * nrec_, w_tmp_, hist_};
    launch_build_records(xyz_dev, zidx_, occ_, nAt_, bg, sb, r.rowptr + (size_t)b0 * rp_stride_, rp_stride_, key_bits_,
                         mask_E_, nconf, st);
}

// jitter + bin + sort + row pointers for the configurations of one batch (slots 0 .. nb-1)
void Engine::prepare_batch(int nb, const float* xyz_k, int set, cudaStream_t st)
{
    if (set < 0) set = act_;
    if (!st) st = st_;
    float* xyzFP = rs_[set].xyzFP;
    if (p_.frPh > 0) {
        // the XORWOW streams are consumed in the global order (k, j) of the single-GPU reference:
        // skip the normals that belong to configurations of other ranks (or other calls)
        long long burn = rng_target_ - rng_pos_;
        if (burn < 0) {
            // a configuration before the current stream position (run_k(k) repeated, k visited out
            // of order): start the streams again, so that configuration (k, j) always sees the
            // draws it has in the reference's (k, j) order
            launch_rng_init(rng_, 3 * nAt_, 1ULL, st);
            rng_pos_ = 0;
            burn = rng_target_;
        }
        launch_atom_jitter(xyzFP, xyz_k, dwf_, nAt_, rng_, burn, nb, st);
        rng_pos_ = rng_target_ + nb;
        rng_target_ = rng_pos_;
    } else {
        for (int b = 0; b < nb; b++)
            CK(cudaMemcpyAsync(xyzFP + (size_t)b * 3 * nAt_, xyz_k, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    bin_and_sort(0, nb, xyzFP, set, st);
}

// Configurations [jb, je) of measurement k in batches of B_, with the atom preparation (jitter, binning,
// radix sort, row pointers: a dozen small launches) of batch i+1 running on the second stream while the
// sweeps of batch i occupy the GPU.  reference_order: configuration j takes the draws it has in the
// reference's (k, j) order (run_k); otherwise the streams simply continue (bench_configs).
void Engine::run_batches(int k, int jb, int je, bool reference_order)
{
    const size_t NN = (size_t)N_ * N_;
    if (je <= jb) return;
    // xyzK_ and the incident wave were enqueued on st_: the preparation stream starts after them; both
    // record sets are free (every earlier use was followed by a synchronisation of st_)
    CK(cudaEventRecord(ev_ready_, st_));
    CK(cudaStreamWaitEvent(st_prep_, ev_ready_, 0));
    auto prepare = [&](int j, int set) {
        const int nb = std::min(B_, je - j);
        if (reference_order) rng_target_ = (long long)k * count_ + j;   // position of configuration (k, j)
        prepare_batch(nb, xyzK_, set, st_prep_);
        CK(cudaEventRecord(ev_prep_[set], st_prep_));
    };
    int set = 0;
    prepare(jb, set);
    for (int j = jb; j < je; j += B_, set ^= 1) {
        const int nb = std::min(B_, je - j);
        if (j + B_ < je) {
            // the other set was last read by the sweeps of batch i-1
            if (j > jb) CK(cudaStreamWaitEvent(st_prep_, ev_used_[set ^ 1], 0));
            prepare(j + B_, set ^ 1);
        }
        CK(cudaStreamWaitEvent(st_, ev_prep_[set], 0));
        act_ = set;
        if (p_.mode != 2 && !p_.doBeamTilt) {
            // psi_in_ is the plane wave: write it directly -- unless the first slice does not read it at all
            // (run_slices_plain: psi = 1, so S6 takes FFT_row(t) straight from D)
            if (!plane_first_slice_) launch_plane_wave_rowspace(Psi_, N_, nb, st_);
        } else {
            for (int b = 0; b < nb; b++)
                CK(cudaMemcpyAsync(Psi_ + (size_t)b * NN, psi_in_, NN * sizeof(cpx), cudaMemcpyDeviceToDevice, st_));
        }
        if (fuse_ctf_ && !ew_) ensure_lens(k);     // read by the last slice's S6
        slice_loop(nb);
        CK(cudaEventRecord(ev_used_[set], st_));
        accumulate_outputs(k, nb);
    }
    act_ = 0;
}

void Engine::run_slices_plain(int nb)
{
    const size_t NN = (size_t)N_ * N_;
    const bool first_full = p_.doBeamTilt && p_.mode == 2;
    const bool fuse = fuse_ctf_ && !ew_;
    // S5 + S6 of one slice; Dp = transmission of configuration 0, d_stride elements between configurations.
    //   first slice of a plane wave: psi = 1, so FFT_row(t psi) is N times what S4 left in D -- no S5, S6 reads D;
    //   last slice with `fuse`: S6 also applies the CTF and writes the filtered waves to W_ (accumulate_outputs).
    auto wave_step = [&](const cpx* Dp, size_t d_stride, int slice) {
        const bool skip_s5 = plane_first_slice_ && slice == 0;
        const bool with_ctf = fuse && slice == p_.m3 - 1;
        if (!skip_s5) launch_multiply_rows(g_, Psi_, Dp, d_stride, nb, first_full && slice == 0, st_);
        if (!skip_s5 && !with_ctf) { launch_propagate_cols(g_, Psi_, Pq_, nb, st_); return; }
        const int img_stride = skip_s5 ? (int)(d_stride / NN) : 1;
        launch_propagate_cols_from(g_, with_ctf ? W_ : Psi_, skip_s5 ? Dp : Psi_, img_stride, img_stride * nb, Pq_, nb,
                                   skip_s5, with_ctf ? lens_ : nullptr, st_);
    };
    // The potential / transmission sweeps S1..S4 run once per PAIR of slices (the two densities
    // share one complex transform); S5/S6 then advance the wave through the two slices in turn.
    for (int s = 0; s < p_.m3; s += 2) {
        const int npair = std::min(2, p_.m3 - s);
        if (npair == 1 && nb % 2 == 0) {
            // odd slice count: the last slices of configurations 2j and 2j + 1 share one complex transform
            // through S1 / S2 / S3 (instead of nb half-empty pairs); S3 writes t of configuration b to D[b]
            potential_pair(s, s, nb / 2, 2, 1);
            launch_transmit_rows(g_, W_, D_, 2, p_.imPot, nb / 2, st_);
            launch_bandlimit_cols(g_, D_, nb, 0, st_);
            wave_step(D_, NN, s);
            break;
        }
        transmission_pair(s, npair, nb, D_);
        for (int p = 0; p < npair; p++) wave_step(D_ + (size_t)p * NN, 2 * NN, s + p);
    }
    if (first_full) launch_zero_outband(Psi_, N_, g_.lo_end, g_.hi_start, nb, st_);
}

void Engine::slice_loop(int nb)
{
    tm_.slices_executed += (long long)p_.m3 * nb;
    // a CUDA graph pays off when the sweeps are launch-bound (small grids, small batches); its
    // capture + instantiation costs about a millisecond, more than it saves on large launches
    if (!opt_.use_graph || (size_t)nb * N_ * N_ > ((size_t)1 << 21)) { run_slices_plain(nb); return; }
    cudaGraphExec_t& graph_ = this->graph_[act_];     // the captured launches carry the record pointers of a set
    int& graph_nb_ = this->graph_nb_[act_];
    long long& graph_launches = graph_launches_[act_];
    const int key = 2 * nb + (fuse_ctf_ && !ew_ ? 1 : 0);     // what the captured launches depend on
    if (!graph_ || graph_nb_ != key) {
        if (graph_) { cudaGraphExecDestroy(graph_); graph_ = nullptr; }
        // first use of each kernel must happen outside capture (function attributes are set there)
        if (!warmed_) { run_slices_plain(nb); warmed_ = true; graph_nb_ = -1; return; }
        cudaGraph_t g = nullptr;
        const long long tally0 = launch_tally;
        CK(cudaStreamBeginCapture(st_, cudaStreamCaptureModeThreadLocal));
        run_slices_plain(nb);
        CK(cudaStreamEndCapture(st_, &g));
        // a capture runs nothing: its kernels count at every launch of the graph
        graph_launches = launch_tally - tally0;
        launch_tally = tally0;
        CK(cudaGraphInstantiate(&graph_, g, 0));
        CK(cudaGraphDestroy(g));
        graph_nb_ = key;
    }
    CK(cudaGraphLaunch(graph_, st_));
    tm_.kernel_launches += graph_launches;
}

// S1 + S2 of a slice pair from the active record set: the potentials of `images` images in W_ (image b: slice s of
// configuration b * cfg_stride, slice s2 of configuration b * cfg_stride + cfg_off2, kernels.cuh)
void Engine::potential_pair(int s, int s2, int images, int cfg_stride, int cfg_off2)
{
    const RecordSet& r = rs_[act_];
    launch_density_rows(g_, A_, r.rowptr, r.cols, r.w, s, s2, nZ_, images, rec_stride_, rp_stride_, st_, cfg_stride, cfg_off2);
    launch_potential_cols(g_, W_, A_, Gq_, r.rowptr, s, s2, nZ_, images, rp_stride_, st_, cfg_stride, cfg_off2);
}

// S1..S4 of slices s, s + 1 (npair = 2) or of slice s alone (npair = 1) of nb configurations: the band-limited
// transmission functions in the [nb][2] stack D
void Engine::transmission_pair(int s, int npair, int nb, cpx* D)
{
    potential_pair(s, npair > 1 ? s + 1 : -1, nb);
    launch_transmit_rows(g_, W_, D, npair, p_.imPot, nb, st_);
    launch_bandlimit_cols(g_, D, nb, npair, st_);
}

// CTF table of measurement k (applyLensFunction, src/multisliceSimulation.cu:614-622), stored [kx][ky]
void Engine::ensure_lens(int k)
{
    if (p_.mode == 0 && lens_k_ != k) {
        launch_lens_table(lens_, N_, lens_params(p_, k, 0), 1.f, st_, /*transposed=*/true);
        lens_k_ = k;
    }
}

void Engine::accumulate_outputs(int k, int nb)
{
    const size_t NN = (size_t)N_ * N_;
    const float alpha = 1.f / ((float)count_);
    ensure_lens(k);
    // exit wave and imaging-mode intensity: the batch is summed inside one launch, in the fixed
    // order b = 0 .. nb-1 (deterministic phonon average)
    if (ew_) {
        RowOpts ro; ro.scale = alpha; ro.band_only_in = true;
        launch_rows_fft_sum(g_, Psi_, ew_, +1, ROW_ACCUM, ro, nb, st_);
    }
    if (p_.mode == 0) {
        // W_ is free after the slice loop: CTF-filtered waves of the whole batch
        // (band columns only where the sweep is pipelined: the wave has no others, and the row sweep below
        // reads none).  With fuse_ctf_ and no exit wave to keep, the last slice's S6 has written them already:
        // IFFT_col(FFT_col(Psi) P lens) = (1/N) IFFT_col(FFT_col(Psi') lens) for Psi' = IFFT_col(FFT_col(Psi) P).
        if (!(fuse_ctf_ && !ew_)) launch_cols_fft(g_, Psi_, W_, -1, COL_MUL_CPX_INV, lens_, 1.f / ((float)N_), nb, st_);
        RowOpts ro; ro.scale = alpha; ro.band_only_in = true;
        launch_rows_fft_sum(g_, W_, I_, +1, ROW_INTENS_ACCUM, ro, nb, st_);
        return;
    }
    for (int b = 0; b < nb; b++) {   // fixed order: deterministic phonon average
        cpx* psi = Psi_ + (size_t)b * NN;
        {
            // diffractionPattern, src/crystalMaker.cu:700-718
            // |fftshift(FFT2 psi)|^2 / N^2: FFT_col(Psi) = FFT2(psi) / N already carries the 1/N
            const float scale = alpha;
            const cpx* src = psi;
            if (p_.doBeamTilt || p_.mode == 1) {
                RowOpts ro; ro.band_only_in = true;
                launch_rows_fft(g_, psi, scratch_, +1, ROW_STORE, ro, 1, st_);
                if (p_.doBeamTilt)
                    launch_tilt_beam(scratch_, N_, p_.d1, p_.d2, p_.lambda, p_.tiltbeam[2 * k],
                                     p_.tiltbeam[2 * k + 1], p_.cst_pi, -1, st_);
                RowOpts r2;
                if (p_.mode == 1) {
                    launch_area_mask_blend(scratch_, N_, p_.dn1, p_.dn2, st_);
                    r2.band_only_out = true;
                    launch_rows_fft(g_, scratch_, scratch_, -1, ROW_STORE, r2, 1, st_);
                    launch_bandlimit_cols(g_, scratch_, 1, 0, st_);
                } else {
                    r2.scale = 1.f / (float)N_;
                    launch_rows_fft(g_, scratch_, scratch_, -1, ROW_STORE, r2, 1, st_);
                }
                src = scratch_;
            }
            launch_cols_fft(g_, src, I_, -1, COL_DP_ACCUM, nullptr, scale, 1, st_);
        }
    }
}

void Engine::run_k(int k)
{
    const Call call(*this);
    PhaseTimer pt;
    if (k < 0 || k >= p_.n3) throw std::runtime_error("measurement index out of range");
    const size_t NN = (size_t)N_ * N_;
    launch_fill_f32(I_, NN, 0.f, st_);
    if (ew_) launch_fill_cpx(ew_, NN, make_float2(0.f, 0.f), st_);
    specimen_k(k);
    make_incident(k);
    run_batches(k, j0_, j1_, true);
    pt.mark("run_k: enqueue");
    CK(cudaStreamSynchronize(st_prep_));
    CK(cudaStreamSynchronize(st_));
    pt.mark("run_k: wait");
}

// Partial sums of other engines (other GPUs of this process, frozen-phonon configurations sharded)
// are added to this engine's accumulators.  All engines must have finished run_k (it synchronises).
void Engine::reduce_from(const std::vector<Engine*>& others)
{
    const Call call(*this);
    if (others.empty()) return;
    if ((int)others.size() > MAX_PEERS) throw std::runtime_error("too many peer engines");
    const size_t NN = (size_t)N_ * N_;
    PeerSources si{}, se{};
    bool direct = true;
    for (Engine* o : others) {
        if (o->N_ != N_) throw std::runtime_error("peer engines must share the grid size");
        if (o->opt_.gpu_index != opt_.gpu_index) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, opt_.gpu_index, o->opt_.gpu_index));
            if (can) {
                const cudaError_t pe = cudaDeviceEnablePeerAccess(o->opt_.gpu_index, 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CK(pe);
                cudaGetLastError();    // clear the sticky "already enabled"
            } else {
                direct = false;
            }
        }
        si.p[si.n++] = o->I_;
        if (ew_ && o->ew_) se.p[se.n++] = reinterpret_cast<const float*>(o->ew_);
    }
    if (direct) {
        launch_peer_sum(I_, si, NN, st_);
        if (ew_ && se.n) launch_peer_sum(reinterpret_cast<float*>(ew_), se, 2 * NN, st_);
    } else {
        // no peer mapping (PCIe boxes without P2P): stage each partial sum through scratch_
        for (Engine* o : others) {
            PeerSources one{};
            one.n = 1;
            CK(cudaMemcpyPeerAsync(scratch_, opt_.gpu_index, o->I_, o->opt_.gpu_index, NN * sizeof(float), st_));
            one.p[0] = reinterpret_cast<const float*>(scratch_);
            launch_peer_sum(I_, one, NN, st_);
            if (ew_ && o->ew_) {
                CK(cudaMemcpyPeerAsync(scratch_, opt_.gpu_index, o->ew_, o->opt_.gpu_index, NN * sizeof(cpx), st_));
                launch_peer_sum(reinterpret_cast<float*>(ew_), one, 2 * NN, st_);
            }
        }
    }
    CK(cudaStreamSynchronize(st_));
}

void Engine::finish_k(int k, float* image_host, float* exitwave_host)
{
    const Call call(*this);
    PhaseTimer pt;
    const size_t NN = (size_t)N_ * N_;
    // addNoiseAndMtf (src/crystalMaker.cu:579-613) + copyMiddleOut
    DetectorParams dp{p_.mtfa, p_.mtfb, p_.mtfc, p_.mtfd, p_.illangle, p_.defoci[k], p_.lambda,
                      p_.d1, p_.d2, p_.cst_pi, p_.mode, fabsf(p_.illangle) > FLT_EPSILON ? 1 : 0};
    const float inv_nn = 1.f / ((float)(N_ * N_));
    RowOpts ri; ri.in_is_real = true;
    launch_rows_fft(g_, I_, scratch_, -1, ROW_STORE, ri, 1, st_);
    if (p_.pD > FLT_EPSILON) {
        // envelope -> back to real space -> Anscombe/Poisson noise -> forward again (:591-603)
        DetectorParams de = dp; de.use_mtf = 0;
        launch_detector_table(det_, N_, de, inv_nn, st_);
        launch_cols_fft(g_, scratch_, scratch_, -1, COL_MUL_REAL_INV, det_, 1.f, 1, st_);
        RowOpts rr;
        launch_rows_fft(g_, scratch_, scratch_, +1, ROW_STORE, rr, 1, st_);
        launch_anscombe_noise(scratch_, NN, p_.pD, noise_rng_, st_);
        launch_rows_fft(g_, scratch_, scratch_, -1, ROW_STORE, rr, 1, st_);
        dp.use_incoherence = 0;   // already applied
    }
    launch_detector_table(det_, N_, dp, inv_nn, st_);
    launch_cols_fft(g_, scratch_, scratch_, -1, COL_MUL_REAL_INV, det_, 1.f, 1, st_);
    RowOpts rc; rc.dn1 = p_.dn1; rc.dn2 = p_.dn2; rc.n1 = p_.n1; rc.n2 = p_.n2;
    launch_rows_fft(g_, scratch_, J_, +1, ROW_CROP_REAL, rc, 1, st_);
    if (image_host)
        CK(cudaMemcpyAsync(image_host, J_, (size_t)p_.n1 * p_.n2 * sizeof(float), cudaMemcpyDeviceToHost, st_));
    if (exitwave_host && ew_)
        CK(cudaMemcpyAsync(exitwave_host, ew_, NN * sizeof(cpx), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    pt.mark("finish_k");
}

// the potential of slice s (records of the active set) in real space, with the absorptive factor -> V_host [m2][m1][2]
void Engine::potential_to_host(int s, float* V_host)
{
    const size_t NN = (size_t)N_ * N_;
    potential_pair(s, -1, 1);
    RowOpts ro;
    launch_rows_fft(g_, W_, scratch_, +1, ROW_STORE, ro, 1, st_);
    launch_absorptive_factor(scratch_, NN, p_.imPot, st_);
    CK(cudaMemcpyAsync(V_host, scratch_, NN * sizeof(cpx), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
}

void Engine::potential_slices(float* out_host)
{
    const Call call(*this);
    // untilted (offset only), phonon-free potential with the original slicing
    // (src/crystalMaker.cu:381-397).  NOTE: the reference leaves this buffer uninitialised when
    // no sub-slicing/phonons/tilt are active; here it is always computed.
    const size_t NN = (size_t)N_ * N_;
    Params save = p_;
    p_.m3 = m3_orig_; p_.d3 = d3_orig_;
    const int nkeys_save = nkeys_, bits_save = key_bits_;
    nkeys_ = m3_orig_ * nZ_ * N_;
    key_bits_ = 0; while ((1LL << key_bits_) <= nkeys_) key_bits_++;
    bin_and_sort(0, 1, xyzTO_);
    for (int s = 0; s < m3_orig_; s++) potential_to_host(s, out_host + (size_t)s * 2 * NN);
    p_ = save; nkeys_ = nkeys_save; key_bits_ = bits_save;
}

// ---------------------------------------------------------------------------------------------
// building blocks for tests / benchmarks
// ---------------------------------------------------------------------------------------------
void Engine::next_jittered_coords(int k, float* xyz_host)
{
    const Call call(*this);
    specimen_k(k);
    if (p_.frPh > 0) { launch_atom_jitter(rs_[act_].xyzFP, xyzK_, dwf_, nAt_, rng_, 0, 1, st_); rng_pos_ += 1; rng_target_ = rng_pos_; }
    else CK(cudaMemcpyAsync(rs_[act_].xyzFP, xyzK_, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st_));
    CK(cudaMemcpyAsync(xyz_host, rs_[act_].xyzFP, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
}

void Engine::bin_tuples(const float* xyz_host, int* bins_host)
{
    const Call call(*this);
    CK(cudaMemcpyAsync(rs_[act_].xyzFP, xyz_host, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    BinGeom bg{N_, N_, p_.m3, nZ_, p_.d1, p_.d2, p_.d3};
    launch_bin_atoms(rs_[act_].xyzFP, zidx_, occ_, nAt_, bg, rs_[act_].keys, rs_[act_].cols, rs_[act_].w, bins_, 1, st_);
    CK(cudaMemcpyAsync(bins_host, bins_, 4 * (size_t)nAt_ * sizeof(int), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
}

void Engine::phase_grating(const float* xyz_host, int s, float* V_host)
{
    const Call call(*this);
    CK(cudaMemcpyAsync(rs_[act_].xyzFP, xyz_host, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    bin_and_sort(0, 1, rs_[act_].xyzFP);
    potential_to_host(s, V_host);
}

void Engine::exit_wave(const float* xyz_host, int k, float* psi_host)
{
    const Call call(*this);
    const size_t NN = (size_t)N_ * N_;
    CK(cudaMemcpyAsync(rs_[act_].xyzFP, xyz_host, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyHostToDevice, st_));
    bin_and_sort(0, 1, rs_[act_].xyzFP);
    make_incident(k);
    CK(cudaMemcpyAsync(Psi_, psi_in_, NN * sizeof(cpx), cudaMemcpyDeviceToDevice, st_));
    const bool ug = opt_.use_graph;
    opt_.use_graph = false;
    slice_loop(1);
    opt_.use_graph = ug;
    RowOpts ro; ro.band_only_in = true; ro.scale = 1.f;
    launch_rows_fft(g_, Psi_, scratch_, +1, ROW_STORE, ro, 1, st_);
    CK(cudaMemcpyAsync(psi_host, scratch_, NN * sizeof(cpx), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
}

double Engine::bench_configs(int k, int configs)
{
    const Call call(*this);
    const size_t NN = (size_t)N_ * N_;
    launch_fill_f32(I_, NN, 0.f, st_);
    if (ew_) launch_fill_cpx(ew_, NN, make_float2(0.f, 0.f), st_);
    specimen_k(k);
    make_incident(k);
    CK(cudaStreamSynchronize(st_));
    CK(cudaEventRecord(ev0_, st_));
    run_batches(k, 0, configs, false);
    CK(cudaEventRecord(ev1_, st_));
    CK(cudaEventSynchronize(ev1_));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    CK(cudaStreamSynchronize(st_prep_));
    tm_.slice_loop_ms += ms;
    return (double)ms;
}

// ---------------------------------------------------------------------------------------------
// STEM probe scan.  FDES itself has no scan (mode 2 = one CBED probe at the grid centre,
// src/multisliceSimulation.cu:572-581); a scan position r_p is that probe shifted periodically by
// a phase ramp in Fourier space, the specimen fixed.  Per frozen-phonon configuration the
// transmission functions of all slices are computed once (S1..S4) and kept in HBM; the probes
// then advance in batches through S5/S6 only, and annular detectors integrate the diffraction
// intensity |FFT2 psi|^2 / N^2 (diffractionPattern, src/crystalMaker.cu:700-718).
// ---------------------------------------------------------------------------------------------
// Checks shared by the scans; the annular detectors as |k|^2 bounds
DetectorRings Engine::stem_rings(int k, int nprobes, int ndet, const float* det_mrad_host, int min_det) const
{
    if (p_.mode != 2) throw std::runtime_error("STEM scan needs mode 2 (convergent probe)");
    if (k < 0 || k >= p_.n3) throw std::runtime_error("measurement index out of range");
    if (nprobes <= 0) throw std::runtime_error("no probe positions");
    if (ndet < min_det || ndet > MAX_DETECTORS) throw std::runtime_error(std::to_string(min_det) + "..8 detectors supported");
    if (p_.doBeamTilt) throw std::runtime_error("STEM scan with beam tilt is not supported");
    DetectorRings rings{};
    rings.n = ndet;
    for (int d = 0; d < ndet; d++) {
        // k^2 = (sin(theta[mrad] * 1e-3) / lambda)^2, the detector convention of src/rwQsc.cu:723-730
        const float a = sinf(det_mrad_host[2 * d] * 1e-3f) / p_.lambda, b = sinf(det_mrad_host[2 * d + 1] * 1e-3f) / p_.lambda;
        rings.in2[d] = a * a;
        rings.out2[d] = b * b;
    }
    return rings;
}

// probe shifts -> shifts (device), zeroed detector sums, incident probe of index k and its column spectrum PSI0 in
// scratch_; returns after the device has taken the host data
void Engine::stem_prepare(int k, int nprobes, const float* xy_host, float* shifts, float* det_out, size_t det_elems)
{
    std::vector<float> sh(2 * (size_t)nprobes);
    for (int i = 0; i < nprobes; i++) {
        sh[2 * i] = xy_host[2 * i] / ((float)N_ * p_.d1);
        sh[2 * i + 1] = xy_host[2 * i + 1] / ((float)N_ * p_.d2);
    }
    CK(cudaMemcpyAsync(shifts, sh.data(), sh.size() * sizeof(float), cudaMemcpyHostToDevice, st_));
    launch_fill_f32(det_out, det_elems, 0.f, st_);
    specimen_k(k);
    make_incident(k);
    // spectrum of the centred probe: PSI0 = FFT_col(psi_in) (scratch_ is free after make_incident)
    launch_cols_fft(g_, psi_in_, scratch_, -1, COL_PLAIN, nullptr, 1.f, 1, st_);
    CK(cudaStreamSynchronize(st_));    // sh goes out of scope
}

// transmission stack of configuration (k, j): the same displacements whenever it is built (rng_target_ re-seeds the
// streams when they are past it)
void Engine::stem_transmission(int k, int j, cpx* tstack)
{
    const size_t NN = (size_t)N_ * N_;
    rng_target_ = (long long)k * count_ + j;
    prepare_batch(1, xyzK_);
    for (int s = 0; s < p_.m3; s += 2) transmission_pair(s, std::min(2, p_.m3 - s), 1, tstack + (size_t)s * NN);
    // (keeping t in real space instead, to save the per-probe inverse row transform of S5,
    // measured SLOWER on B200: 8.3k vs 9.5k probes/s at 512^2 -- the transform hides the
    // latency of the wave loads)
}

// nb probes at shifts through every slice of tstack: exit waves in Psi_
void Engine::stem_probes(const float* shifts, int nb, const cpx* tstack)
{
    const size_t NN = (size_t)N_ * N_;
    launch_probe_cols(g_, Psi_, scratch_, shifts, nb, st_);
    for (int s = 0; s < p_.m3; s++) {
        launch_multiply_rows(g_, Psi_, tstack + (size_t)s * NN, 0, nb, false, st_);
        launch_propagate_cols(g_, Psi_, Pq_, nb, st_);
    }
    tm_.slices_executed += (long long)p_.m3 * nb;
}

void Engine::stem_scan(int k, int nprobes, const float* xy_host, int ndet, const float* det_mrad_host,
                       float* out_host, double* loop_ms)
{
    const Call call(*this);
    const DetectorRings rings = stem_rings(k, nprobes, ndet, det_mrad_host, 1);
    const size_t NN = (size_t)N_ * N_;
    // device scratch of this call: transmission stack, probe shifts, detector sums
    const int tiles = detector_tiles(g_);
    cpx* tstack = nullptr; float *shifts = nullptr, *out = nullptr, *partial = nullptr;
    ArenaPlan plan;
    plan.add(tstack, ((size_t)p_.m3 + 1) * NN);
    plan.add(shifts, 2 * (size_t)nprobes);
    plan.add(out, (size_t)nprobes * ndet);
    plan.add(partial, (size_t)B_ * tiles * MAX_DETECTORS);
    void* block = pool_acquire(plan.total(), opt_.gpu_index);
    plan.assign(block);
    try {
        stem_prepare(k, nprobes, xy_host, shifts, out, (size_t)nprobes * ndet);
        CK(cudaEventRecord(ev0_, st_));
        const float weight = 1.f / (float)count_;
        for (int j = j0_; j < j1_; j++) {
            stem_transmission(k, j, tstack);
            for (int i0 = 0; i0 < nprobes; i0 += B_) {
                const int nb = std::min(B_, nprobes - i0);
                stem_probes(shifts + 2 * (size_t)i0, nb, tstack);
                launch_detector_cols(g_, Psi_, partial, out + (size_t)i0 * ndet, rings, p_.d1, p_.d2, weight, nb, st_);
            }
        }
        CK(cudaEventRecord(ev1_, st_));
        CK(cudaMemcpyAsync(out_host, out, (size_t)nprobes * ndet * sizeof(float), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        if (loop_ms) { float ms = 0.f; CK(cudaEventElapsedTime(&ms, ev0_, ev1_)); *loop_ms = ms; }
    } catch (...) {
        cudaStreamSynchronize(st_);
        pool_release(block);
        throw;
    }
    pool_release(block);
}

// ---------------------------------------------------------------------------------------------
// 4D-STEM: the diffraction pattern of every probe, fftshifted, cropped to a centred window of Q x Q pixels and
// binned bin x bin.  A whole data set does not fit the device (256^2 probes x 342^2 pixels x 4 B = 30 GB at 512^2),
// so the raster runs in passes of probes_per_pass probes; a pass rebuilds the transmission stack of every
// configuration (S1..S4 are a small share of a pass: one stack per configuration against m3 x (S5, S6) per probe).
// Finished passes go to the host from the other of two device pass buffers while the next pass computes: in chunks
// through two pinned buffers on two copy streams, each chunk copied on to its place in the caller's array by a
// host function of its stream.
// ---------------------------------------------------------------------------------------------
int stem4d_window(int N, int window, int bin)
{
    if (N < 1) throw std::runtime_error("grid size must be positive");
    if (bin < 1) throw std::runtime_error("4D-STEM bin must be >= 1");
    if (window < 0) throw std::runtime_error("4D-STEM window must be >= 0 (0: the band limit)");
    if (window == 0) {
        // kb: the largest |i| the band limit keeps on an axis (zeroHighFreq's float test, src/multisliceSimulation.cu:225-250;
        // the same loop as make_sweep_geom).  Window pixel q holds frequency q - Q/2: an even Q covers [-Q/2, Q/2 - 1],
        // an odd Q [-(Q-1)/2, (Q-1)/2].
        int kb = 0;
        const float mind = (float)N;
        while (kb + 1 <= N / 2 && !(((float)((kb + 1) * (kb + 1)) * 9.f / (mind * mind)) > 1.f)) kb++;
        int Q = 2 * kb + 1 + (N % 2 == 0 ? 1 : 0);
        while (Q <= N && Q % bin != 0) Q += 2;
        if (Q > N)
            throw std::runtime_error("4D-STEM: no window of N's parity (N = " + std::to_string(N) + ") that is a multiple of bin " +
                                     std::to_string(bin) + " holds the band limit");
        return Q;
    }
    if (window > N) throw std::runtime_error("4D-STEM window " + std::to_string(window) + " larger than the grid (" + std::to_string(N) + ")");
    if ((N - window) % 2 != 0)
        throw std::runtime_error("4D-STEM window " + std::to_string(window) + " must have the parity of the grid size " + std::to_string(N) +
                                 " (a whole-pixel centred crop)");
    if (window % bin != 0)
        throw std::runtime_error("4D-STEM window " + std::to_string(window) + " is not a multiple of bin " + std::to_string(bin));
    return window;
}

int Engine::stem_4d_probes_per_pass(int nprobes, int window, int bin)
{
    const Call call(*this);
    const int S = stem4d_window(N_, window, bin) / bin;
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    // the two pass buffers: at most about a quarter of the free memory
    const size_t per_probe = 2 * (size_t)S * S * sizeof(float);
    return (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(nprobes, 1), fr / 4 / per_probe));
}

namespace {
struct HostCopy { float* dst; const float* src; size_t bytes; };
void CUDART_CB host_copy(void* p)
{
    const HostCopy* c = static_cast<const HostCopy*>(p);
    memcpy(c->dst, c->src, c->bytes);
}
// copy streams, events and pinned chunks of one 4D scan; the destructor waits for every copy
struct PassCopies {
    static constexpr size_t CHUNK = (size_t)64 << 20;    // bytes per pinned buffer
    cudaStream_t st[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    float* pin[2] = {nullptr, nullptr};
    PassCopies()
    {
        for (int i = 0; i < 2; i++) {
            CK(cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
            for (int q = 0; q < 2; q++) CK(cudaEventCreateWithFlags(&copied[i][q], cudaEventDisableTiming));
            CK(cudaHostAlloc(reinterpret_cast<void**>(&pin[i]), CHUNK, cudaHostAllocDefault));
        }
    }
    ~PassCopies()
    {
        for (int i = 0; i < 2; i++) {
            if (st[i]) { cudaStreamSynchronize(st[i]); cudaStreamDestroy(st[i]); }
            if (done[i]) cudaEventDestroy(done[i]);
            for (int q = 0; q < 2; q++) if (copied[i][q]) cudaEventDestroy(copied[i][q]);
            if (pin[i]) cudaFreeHost(pin[i]);
        }
    }
    PassCopies(const PassCopies&) = delete;
    PassCopies& operator=(const PassCopies&) = delete;
};
}  // namespace

void Engine::stem_scan_4d(int k, int nprobes, const float* xy_host, int window, int bin, int ndet, const float* det_mrad_host,
                          int probes_per_pass, float* out_pattern_host, float* out_det_host, double* loop_ms)
{
    const Call call(*this);
    const DetectorRings rings = stem_rings(k, nprobes, ndet, det_mrad_host, 0);
    const int Q = stem4d_window(N_, window, bin);
    const size_t NN = (size_t)N_ * N_, QQ = (size_t)Q * Q, SS = (size_t)(Q / bin) * (Q / bin);
    if (probes_per_pass < 0) throw std::runtime_error("probes_per_pass must be >= 0 (0: automatic)");
    if (!out_pattern_host || (ndet > 0 && !out_det_host)) throw std::runtime_error("4D-STEM output array is NULL");
    const int ppp = std::min(nprobes, probes_per_pass > 0 ? probes_per_pass : stem_4d_probes_per_pass(nprobes, window, bin));
    const int tiles = detector_tiles(g_);
    cpx* tstack = nullptr;
    float *shifts = nullptr, *det = nullptr, *partial = nullptr, *scratch4d = nullptr, *pass[2] = {nullptr, nullptr};
    ArenaPlan plan;
    plan.add(tstack, ((size_t)p_.m3 + 1) * NN);
    plan.add(shifts, 2 * (size_t)nprobes);
    plan.add(det, (size_t)nprobes * ndet);
    plan.add(partial, (size_t)B_ * tiles * MAX_DETECTORS);
    plan.add(scratch4d, (size_t)B_ * QQ);
    for (float*& p : pass) plan.add(p, (size_t)ppp * SS);
    void* block = pool_acquire(plan.total(), opt_.gpu_index);
    plan.assign(block);
    const int npass = (nprobes + ppp - 1) / ppp;
    const size_t chunk = PassCopies::CHUNK / sizeof(float);
    std::vector<HostCopy> jobs;      // read by the host functions: no reallocation while they are queued
    jobs.reserve((size_t)npass * (((size_t)ppp * SS + chunk - 1) / chunk));
    try {
        PassCopies pc;
        stem_prepare(k, nprobes, xy_host, shifts, det, (size_t)nprobes * ndet);
        // the pixels outside the band columns are never written by the 4D sweep
        launch_fill_f32(scratch4d, (size_t)B_ * QQ, 0.f, st_);
        CK(cudaEventRecord(ev0_, st_));
        const float weight = 1.f / (float)count_;
        size_t c = 0;
        for (int pi = 0; pi < npass; pi++) {
            const int s = pi & 1, p0 = pi * ppp, np = std::min(ppp, nprobes - p0);
            if (pi >= 2)      // pass buffer s still on its way to the host (pass pi - 2)
                for (int q = 0; q < 2; q++) CK(cudaStreamWaitEvent(st_, pc.copied[s][q], 0));
            launch_fill_f32(pass[s], (size_t)np * SS, 0.f, st_);
            for (int j = j0_; j < j1_; j++) {
                stem_transmission(k, j, tstack);
                for (int i0 = 0; i0 < np; i0 += B_) {
                    const int nb = std::min(B_, np - i0);
                    stem_probes(shifts + 2 * (size_t)(p0 + i0), nb, tstack);
                    launch_detector4d_cols(g_, Psi_, scratch4d, pass[s] + (size_t)i0 * SS, Q, bin, weight, nb, st_);
                    if (ndet > 0)
                        launch_detector_cols(g_, Psi_, partial, det + (size_t)(p0 + i0) * ndet, rings, p_.d1, p_.d2, weight, nb, st_);
                }
            }
            CK(cudaEventRecord(pc.done[s], st_));
            for (int q = 0; q < 2; q++) CK(cudaStreamWaitEvent(pc.st[q], pc.done[s], 0));
            const size_t total = (size_t)np * SS;
            for (size_t off = 0; off < total; off += chunk, c++) {
                const int q = (int)(c & 1);
                const size_t n = std::min(chunk, total - off);
                CK(cudaMemcpyAsync(pc.pin[q], pass[s] + off, n * sizeof(float), cudaMemcpyDeviceToHost, pc.st[q]));
                jobs.push_back({out_pattern_host + (size_t)p0 * SS + off, pc.pin[q], n * sizeof(float)});
                CK(cudaLaunchHostFunc(pc.st[q], host_copy, &jobs.back()));
            }
            for (int q = 0; q < 2; q++) CK(cudaEventRecord(pc.copied[s][q], pc.st[q]));
        }
        CK(cudaEventRecord(ev1_, st_));
        if (ndet > 0) CK(cudaMemcpyAsync(out_det_host, det, (size_t)nprobes * ndet * sizeof(float), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        for (int q = 0; q < 2; q++) CK(cudaStreamSynchronize(pc.st[q]));
        if (loop_ms) { float ms = 0.f; CK(cudaEventElapsedTime(&ms, ev0_, ev1_)); *loop_ms = ms; }
    } catch (...) {
        cudaStreamSynchronize(st_);
        pool_release(block);
        throw;
    }
    pool_release(block);
}

// Each of the six sweeps launched `reps` times back to back on the buffers of a prepared batch,
// bracketed by CUDA events on the engine's stream: ms6[i] = average launch duration of S(i+1).
void Engine::time_sweeps(int k, int nb, int reps, float* ms6)
{
    const Call call(*this);
    const size_t NN = (size_t)N_ * N_;
    nb = std::max(1, std::min(nb, B_));
    CK(cudaMemcpyAsync(xyzK_, xyzTO_, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st_));
    make_incident(k);
    for (int b = 0; b < nb; b++) {
        float* fp = rs_[act_].xyzFP + (size_t)b * 3 * nAt_;
        CK(cudaMemcpyAsync(fp, xyzK_, 3 * (size_t)nAt_ * sizeof(float), cudaMemcpyDeviceToDevice, st_));
        bin_and_sort(b, 1, fp);
        CK(cudaMemcpyAsync(Psi_ + (size_t)b * NN, psi_in_, NN * sizeof(cpx), cudaMemcpyDeviceToDevice, st_));
    }
    // a slice pair in the middle of the specimen; S1..S4 are timed on the pair and reported per
    // slice (half), S5/S6 on one slice
    const int s = std::max(0, (p_.m3 / 2) & ~1);
    const int npair = std::min(2, p_.m3 - s);
    const int s2 = npair > 1 ? s + 1 : -1;
    for (int i = 0; i < 6; i++) {
        for (int r = -1; r < reps; r++) {   // r = -1: untimed warm-up launch
            if (r == 0) CK(cudaEventRecord(ev0_, st_));
            switch (i) {
                case 0: launch_density_rows(g_, A_, rs_[act_].rowptr, rs_[act_].cols, rs_[act_].w, s, s2, nZ_, nb, rec_stride_, rp_stride_, st_); break;
                case 1: launch_potential_cols(g_, W_, A_, Gq_, rs_[act_].rowptr, s, s2, nZ_, nb, rp_stride_, st_); break;
                case 2: launch_transmit_rows(g_, W_, D_, npair, p_.imPot, nb, st_); break;
                case 3: launch_bandlimit_cols(g_, D_, nb, npair, st_); break;
                case 4: launch_multiply_rows(g_, Psi_, D_, 2 * NN, nb, false, st_); break;
                case 5: launch_propagate_cols(g_, Psi_, Pq_, nb, st_); break;
            }
        }
        CK(cudaEventRecord(ev1_, st_));
        CK(cudaEventSynchronize(ev1_));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev0_, ev1_));
        ms6[i] = ms / (float)reps / (i < 4 ? (float)npair : 1.f);   // per slice
    }
}

}  // namespace fdes
