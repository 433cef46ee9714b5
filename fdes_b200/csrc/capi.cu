// fdes_b200 -- C ABI (include/fdes_b200.h): the drop-in FDES() symbol of the reference
// (src/FDESExport.cu:59-178) and the session API over the engine.
#include "../../include/fdes_b200.h"
#include "engine.h"
#include "emd.h"
#include "qsc.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <memory>
#include <stdexcept>
#include <vector>
#include <algorithm>
#include <string>
#include <chrono>
#include <climits>
#include <thread>
#include <exception>

using namespace fdes;

std::vector<int> fdes_b200_gpu_list(const char* spec, int first);

// A session owns one engine per GPU it runs on.  With several GPUs the work of a run is sharded
// over the engines of this ONE process (one host thread per device while they compute):
//   SHARD_CONFIGS   frozen-phonon configurations j of every measurement k (src/crystalMaker.cu:332);
//                   the partial sums are reduced onto the first device (Engine::reduce_from)
//   SHARD_REPLICAS  every engine holds the whole problem: measurements k (tilt / defocus series,
//                   src/crystalMaker.cu:324) or STEM probe positions are dealt out, nothing to reduce
enum { SHARD_NONE = 0, SHARD_CONFIGS = 1, SHARD_REPLICAS = 2 };
struct fdes_b200_sim {
    std::vector<std::unique_ptr<Engine>> engs;
    Engine* eng = nullptr;   // engs[0]: the engine of single-GPU sessions, the reduction root otherwise
    int shard = SHARD_NONE;
    Params params;   // as read (before sub-slicing)
    Atoms atoms;
    int m3_orig = 1;
};

// f(r) for r = 0 .. n-1 on n host threads (r = 0 on the caller's); the first exception is rethrown
template <class F>
static void parallel_for(int n, F f)
{
    if (n <= 1) { if (n == 1) f(0); return; }
    std::vector<std::exception_ptr> err(n);
    std::vector<std::thread> th;
    th.reserve(n - 1);
    for (int r = 1; r < n; r++)
        th.emplace_back([&, r] { try { f(r); } catch (...) { err[r] = std::current_exception(); } });
    try { f(0); } catch (...) { err[0] = std::current_exception(); }
    for (auto& t : th) t.join();
    for (auto& e : err) if (e) std::rethrow_exception(e);
}

static thread_local std::string g_err;

#define API_TRY try {
#define API_CATCH(ret)                                                                           \
    }                                                                                            \
    catch (const std::exception& e) { g_err = e.what(); return ret; }                            \
    catch (...) { g_err = "unknown error"; return ret; }

extern "C" {

const char* fdes_b200_last_error(void) { return g_err.c_str(); }
int fdes_b200_version(void) { return 100; }

int fdes_b200_parse_cnf(const char* cnf_path, int* dims, float* scalars, float* per_k,
                        float* atoms6_out, int max_atoms)
{
    API_TRY
    if (!cnf_path) throw std::runtime_error("cnf_path is NULL");
    Params p;
    Atoms at;
    if (!read_input(cnf_path, p, &at, false)) throw std::runtime_error(std::string("cannot read ") + cnf_path);
    set_sub_slices(p, sub_slice_ratio(p.d3, p.subSlTh));
    if (dims) {
        dims[0] = p.n1; dims[1] = p.n2; dims[2] = p.n3; dims[3] = p.m1; dims[4] = p.m2; dims[5] = p.m3;
        dims[6] = at.size(); dims[7] = (int)list_of_elements(at.Z).size(); dims[8] = p.frPh; dims[9] = p.mode;
    }
    if (scalars) {
        scalars[0] = p.lambda; scalars[1] = p.sigma; scalars[2] = p.gamma; scalars[3] = p.d1;
        scalars[4] = p.d2; scalars[5] = p.d3; scalars[6] = p.E0; scalars[7] = p.imPot;
    }
    if (per_k)
        for (int k = 0; k < p.n3; k++) {
            per_k[5 * k + 0] = p.tiltspec[2 * k]; per_k[5 * k + 1] = p.tiltspec[2 * k + 1];
            per_k[5 * k + 2] = p.tiltbeam[2 * k]; per_k[5 * k + 3] = p.tiltbeam[2 * k + 1];
            per_k[5 * k + 4] = p.defoci[k];
        }
    if (atoms6_out)
        for (int i = 0; i < at.size() && i < max_atoms; i++) {
            float* a = atoms6_out + 6 * (size_t)i;
            a[0] = (float)at.Z[i]; a[1] = at.xyz[3 * i]; a[2] = at.xyz[3 * i + 1]; a[3] = at.xyz[3 * i + 2];
            a[4] = at.dwf[i]; a[5] = at.occ[i];
        }
    return at.size();
    API_CATCH(-1)
}

int fdes_b200_write_used_cnf(const char* input_path, const char* out_path)
{
    API_TRY
    if (!input_path || !out_path) throw std::runtime_error("path is NULL");
    Params p;
    Atoms at;
    if (!read_input(input_path, p, &at, false)) throw std::runtime_error(std::string("cannot read ") + input_path);
    if (!write_cnf(out_path, p, at, 0)) throw std::runtime_error(std::string("cannot write ") + out_path);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_qsc_scan(const char* qsc_path, int* nxy, float* xy_host, int max_probes, float* det_mrad_host,
                       int max_det)
{
    API_TRY
    if (!qsc_path) throw std::runtime_error("qsc_path is NULL");
    QscScan sc;
    if (!read_qsc_scan(qsc_path, sc)) throw std::runtime_error(std::string("cannot read ") + qsc_path);
    const int np = sc.nx * sc.ny, nd = (int)sc.det_mrad.size() / 2;
    if (nxy) { nxy[0] = sc.nx; nxy[1] = sc.ny; }
    if (xy_host) memcpy(xy_host, sc.xy.data(), sizeof(float) * 2 * (size_t)std::min(np, max_probes));
    if (det_mrad_host) memcpy(det_mrad_host, sc.det_mrad.data(), sizeof(float) * 2 * (size_t)std::min(nd, max_det));
    return nd;
    API_CATCH(-1)
}

int fdes_b200_write_emd(const char* input_path, const char* emd_path, const float* image_host,
                        const float* potential_host, int pot_slices, const float* exitwave_host)
{
    API_TRY
    if (!input_path || !emd_path) throw std::runtime_error("path is NULL");
    Params p;
    Atoms at;
    if (!read_input(input_path, p, &at, false)) throw std::runtime_error(std::string("cannot read ") + input_path);
    if (!write_emd(emd_path, p, at, image_host, potential_host, pot_slices, exitwave_host))
        throw std::runtime_error(std::string("cannot write ") + emd_path);
    return 0;
    API_CATCH(-1)
}

static std::unique_ptr<fdes_b200_sim> read_session(const char* cnf_path, const float* atoms6, int numAtoms)
{
    auto sim = std::make_unique<fdes_b200_sim>();
    if (!cnf_path) throw std::runtime_error("cnf_path is NULL");
    if (!read_input(cnf_path, sim->params, &sim->atoms, atoms6 != nullptr))
        throw std::runtime_error(std::string("cannot read ") + cnf_path);
    if (atoms6) {
        if (numAtoms <= 0) throw std::runtime_error("numAtoms must be positive");
        atoms_from_array(atoms6, numAtoms, sim->atoms);
    }
    sim->params.nAt = sim->atoms.size();
    sim->m3_orig = sim->params.m3;
    return sim;
}

fdes_b200_sim* fdes_b200_open_cnf(const char* cnf_path, const float* atoms6, int numAtoms,
                                  int gpu_index, int batch, int rank, int world, int want_exitwave)
{
    API_TRY
    auto sim = read_session(cnf_path, atoms6, numAtoms);
    EngineOptions opt;
    opt.gpu_index = gpu_index; opt.batch = batch; opt.rank = rank; opt.world = world;
    opt.want_exitwave = want_exitwave != 0;
    sim->engs.push_back(std::make_unique<Engine>(sim->params, sim->atoms, opt));
    sim->eng = sim->engs[0].get();
    return sim.release();
    API_CATCH(nullptr)
}

fdes_b200_sim* fdes_b200_open_multi(const char* cnf_path, const float* atoms6, int numAtoms,
                                    const int* gpu_indices, int ngpus, int batch, int want_exitwave)
{
    API_TRY
    if (!gpu_indices || ngpus < 1) throw std::runtime_error("need at least one GPU index");
    if (ngpus > MAX_PEERS + 1) throw std::runtime_error("at most 16 GPUs per session");
    auto sim = read_session(cnf_path, atoms6, numAtoms);
    const Params& p = sim->params;
    const int count = p.frPh > 0 ? p.frPh : 1;
    int n = 1;
    if (ngpus > 1 && count >= 2) { sim->shard = SHARD_CONFIGS; n = std::min(ngpus, count); }
    else if (ngpus > 1 && (p.n3 >= 2 || p.mode == 2)) { sim->shard = SHARD_REPLICAS; n = ngpus; }
    sim->engs.resize(n);
    fdes_b200_sim* raw = sim.get();
    parallel_for(n, [&](int r) {
        EngineOptions opt;
        opt.gpu_index = gpu_indices[r]; opt.batch = batch;
        opt.rank = raw->shard == SHARD_CONFIGS ? r : 0;
        opt.world = raw->shard == SHARD_CONFIGS ? n : 1;
        opt.want_exitwave = want_exitwave != 0;
        raw->engs[r] = std::make_unique<Engine>(raw->params, raw->atoms, opt);
    });
    sim->eng = sim->engs[0].get();
    return sim.release();
    API_CATCH(nullptr)
}

int fdes_b200_num_gpus(const fdes_b200_sim* sim) { return sim ? (int)sim->engs.size() : -1; }

void fdes_b200_close(fdes_b200_sim* sim) { delete sim; }

int fdes_b200_get_dims(const fdes_b200_sim* sim, int* d)
{
    API_TRY
    const Params& p = sim->eng->params();
    d[0] = p.n1; d[1] = p.n2; d[2] = p.n3; d[3] = p.m1; d[4] = p.m2; d[5] = p.m3;
    d[6] = sim->atoms.size(); d[7] = sim->eng->num_species(); d[8] = sim->eng->configs_total();
    d[9] = sim->eng->batch();
    return 0;
    API_CATCH(-1)
}

int fdes_b200_get_scalars(const fdes_b200_sim* sim, float* s)
{
    API_TRY
    const Params& p = sim->eng->params();
    s[0] = p.lambda; s[1] = p.sigma; s[2] = p.gamma; s[3] = p.d1; s[4] = p.d2; s[5] = p.d3;
    s[6] = p.E0; s[7] = p.imPot;
    return 0;
    API_CATCH(-1)
}

int fdes_b200_set_accumulators(fdes_b200_sim* sim, float* intensity_dev, float* exitwave_dev)
{
    API_TRY
    sim->eng->set_accumulators(intensity_dev, reinterpret_cast<cpx*>(exitwave_dev));
    return 0;
    API_CATCH(-1)
}

int fdes_b200_run_k(fdes_b200_sim* sim, int k)
{
    API_TRY
    sim->eng->run_k(k);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_finish_k(fdes_b200_sim* sim, int k, float* image_host, float* exitwave_host)
{
    API_TRY
    sim->eng->finish_k(k, image_host, exitwave_host);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_simulate(fdes_b200_sim* sim, float* image_host, float* exitwave_host)
{
    API_TRY
    const Params& p = sim->eng->params();
    const size_t n12 = (size_t)p.n1 * p.n2, m12 = (size_t)p.m1 * p.m2;
    const int n = (int)sim->engs.size();
    auto img_k = [&](int k) { return image_host ? image_host + k * n12 : nullptr; };
    auto ew_k = [&](int k) { return exitwave_host ? exitwave_host + 2 * k * m12 : nullptr; };
    if (n > 1 && sim->shard == SHARD_CONFIGS) {
        // every device runs its configurations of measurement k; device 0 adds the partial sums
        // (peer reads over NVLink) and runs the detector tail, as the reference does once per k
        // after its j loop (src/crystalMaker.cu:332-372)
        std::vector<Engine*> others;
        for (int r = 1; r < n; r++) others.push_back(sim->engs[r].get());
        for (int k = 0; k < p.n3; k++) {
            parallel_for(n, [&](int r) { sim->engs[r]->run_k(k); });
            sim->eng->reduce_from(others);
            sim->eng->finish_k(k, img_k(k), ew_k(k));
        }
    } else if (n > 1 && sim->shard == SHARD_REPLICAS && p.n3 > 1) {
        parallel_for(n, [&](int r) {
            for (int k = r; k < p.n3; k += n) {
                sim->engs[r]->run_k(k);
                sim->engs[r]->finish_k(k, img_k(k), ew_k(k));
            }
        });
    } else {
        for (int k = 0; k < p.n3; k++) {
            sim->eng->run_k(k);
            sim->eng->finish_k(k, img_k(k), ew_k(k));
        }
    }
    return 0;
    API_CATCH(-1)
}

int fdes_b200_potential_slices_count(const fdes_b200_sim* sim) { return sim ? sim->m3_orig : -1; }

int fdes_b200_potential(fdes_b200_sim* sim, float* out_host)
{
    API_TRY
    sim->eng->potential_slices(out_host);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_jitter_next(fdes_b200_sim* sim, int k, float* xyz_host)
{
    API_TRY
    sim->eng->next_jittered_coords(k, xyz_host);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_bin_atoms(fdes_b200_sim* sim, const float* xyz_host, int* bins_host)
{
    API_TRY
    sim->eng->bin_tuples(xyz_host, bins_host);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_phase_grating(fdes_b200_sim* sim, const float* xyz_host, int slice, float* V_host)
{
    API_TRY
    if (slice < 0 || slice >= sim->eng->params().m3) throw std::runtime_error("slice out of range");
    sim->eng->phase_grating(xyz_host, slice, V_host);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_exit_wave(fdes_b200_sim* sim, const float* xyz_host, int k, float* psi_host)
{
    API_TRY
    sim->eng->exit_wave(xyz_host, k, psi_host);
    return 0;
    API_CATCH(-1)
}

double fdes_b200_bench_configs(fdes_b200_sim* sim, int k, int configs)
{
    API_TRY
    return sim->eng->bench_configs(k, configs);
    API_CATCH(-1.0)
}

double fdes_b200_stem_scan(fdes_b200_sim* sim, int k, int nprobes, const float* xy_host, int ndet,
                           const float* det_mrad_host, float* out_host)
{
    API_TRY
    const int n = (int)sim->engs.size();
    if (n > 1 && nprobes > 0 && ndet > 0) {
        std::vector<double> ms(n, 0.0);
        if (sim->shard == SHARD_CONFIGS) {
            // every device scans all positions with its share of the frozen-phonon configurations
            // (weights 1/count inside); the detector signals are summed here in device order
            std::vector<std::vector<float>> part(n);
            parallel_for(n, [&](int r) {
                part[r].resize((size_t)nprobes * ndet);
                sim->engs[r]->stem_scan(k, nprobes, xy_host, ndet, det_mrad_host, part[r].data(), &ms[r]);
            });
            for (size_t i = 0; i < (size_t)nprobes * ndet; i++) {
                float s = part[0][i];
                for (int r = 1; r < n; r++) s += part[r][i];
                out_host[i] = s;
            }
        } else {
            // replicas: contiguous ranges of the raster per device, gathered in place
            parallel_for(n, [&](int r) {
                const int i0 = (int)((long long)nprobes * r / n), i1 = (int)((long long)nprobes * (r + 1) / n);
                if (i1 > i0)
                    sim->engs[r]->stem_scan(k, i1 - i0, xy_host + 2 * (size_t)i0, ndet, det_mrad_host,
                                            out_host + (size_t)i0 * ndet, &ms[r]);
            });
        }
        return *std::max_element(ms.begin(), ms.end());
    }
    double ms = 0.0;
    sim->eng->stem_scan(k, nprobes, xy_host, ndet, det_mrad_host, out_host, &ms);
    return ms;
    API_CATCH(-1.0)
}

int fdes_b200_stem_4d_side(int N, int window, int bin)
{
    API_TRY
    return stem4d_window(N, window, bin) / bin;
    API_CATCH(-1)
}

double fdes_b200_stem_scan_4d(fdes_b200_sim* sim, int k, int nprobes, const float* xy_host, int window, int bin, int ndet,
                              const float* det_mrad_host, int probes_per_pass, float* patterns_host, float* det_out_host)
{
    API_TRY
    if (!patterns_host || (ndet > 0 && !det_out_host)) throw std::runtime_error("4D-STEM output array is NULL");
    const int n = (int)sim->engs.size();
    if (n > 1 && nprobes > 0) {
        const int side = stem4d_window(sim->eng->grid(), window, bin) / bin;
        const size_t SS = (size_t)side * side;
        std::vector<double> ms(n, 0.0);
        if (sim->shard == SHARD_CONFIGS) {
            // every device computes each pass with its share of the frozen-phonon configurations (weights 1/count
            // inside); the passes are summed here in device order, so that the host holds one pass per device
            if (probes_per_pass < 0) throw std::runtime_error("probes_per_pass must be >= 0 (0: automatic)");
            int ppp = probes_per_pass > 0 ? std::min(probes_per_pass, nprobes) : nprobes;
            if (probes_per_pass == 0)
                for (auto& e : sim->engs) ppp = std::min(ppp, e->stem_4d_probes_per_pass(nprobes, window, bin));
            std::vector<std::vector<float>> part(n), dpart(n);
            for (int p0 = 0; p0 < nprobes; p0 += ppp) {
                const int np = std::min(ppp, nprobes - p0);
                parallel_for(n, [&](int r) {
                    part[r].resize((size_t)np * SS);
                    dpart[r].resize((size_t)np * ndet);
                    double t = 0.0;
                    sim->engs[r]->stem_scan_4d(k, np, xy_host + 2 * (size_t)p0, window, bin, ndet, det_mrad_host, np, part[r].data(),
                                               dpart[r].data(), &t);
                    ms[r] += t;
                });
                for (size_t i = 0; i < (size_t)np * SS; i++) {
                    float s = part[0][i];
                    for (int r = 1; r < n; r++) s += part[r][i];
                    patterns_host[(size_t)p0 * SS + i] = s;
                }
                for (size_t i = 0; i < (size_t)np * ndet; i++) {
                    float s = dpart[0][i];
                    for (int r = 1; r < n; r++) s += dpart[r][i];
                    det_out_host[(size_t)p0 * ndet + i] = s;
                }
            }
        } else {
            // replicas: contiguous ranges of the raster per device, written in place
            parallel_for(n, [&](int r) {
                const int i0 = (int)((long long)nprobes * r / n), i1 = (int)((long long)nprobes * (r + 1) / n);
                if (i1 > i0)
                    sim->engs[r]->stem_scan_4d(k, i1 - i0, xy_host + 2 * (size_t)i0, window, bin, ndet, det_mrad_host, probes_per_pass,
                                               patterns_host + (size_t)i0 * SS, det_out_host ? det_out_host + (size_t)i0 * ndet : nullptr,
                                               &ms[r]);
            });
        }
        return *std::max_element(ms.begin(), ms.end());
    }
    double ms = 0.0;
    sim->eng->stem_scan_4d(k, nprobes, xy_host, window, bin, ndet, det_mrad_host, probes_per_pass, patterns_host, det_out_host, &ms);
    return ms;
    API_CATCH(-1.0)
}

int fdes_b200_time_sweeps(fdes_b200_sim* sim, int k, int batch, int reps, float* ms6)
{
    API_TRY
    if (reps < 1) throw std::runtime_error("reps must be >= 1");
    sim->eng->time_sweeps(k, batch, reps, ms6);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_get_counters(fdes_b200_sim* sim, long long* c, int reset)
{
    API_TRY
    const EngineTimings& t = sim->eng->timings();
    c[0] = t.slices_executed; c[1] = t.kernel_launches; c[2] = sim->eng->band_columns(); c[3] = 0;
    if (reset) sim->eng->reset_timings();
    return 0;
    API_CATCH(-1)
}

int fdes_b200_fft2d(float* data_host, int N, int dir, int gpu_index)
{
    API_TRY
    if (!fft_size_supported(N)) throw std::runtime_error("unsupported FFT size");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device");
    CK(cudaSetDevice(gpu_index));
    const size_t NN = (size_t)N * N;
    cpx *d = nullptr, *tw = nullptr;
    CK(cudaMalloc(&d, NN * sizeof(cpx)));
    const std::vector<cpx> h = make_twiddles(N);
    CK(cudaMalloc(&tw, h.size() * sizeof(cpx)));
    CK(cudaMemcpy(tw, h.data(), h.size() * sizeof(cpx), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d, data_host, NN * sizeof(cpx), cudaMemcpyHostToDevice));
    SweepGeom g{N, N, N, tw};
    RowOpts ro;
    launch_rows_fft(g, d, d, dir, ROW_STORE, ro, 1, 0);
    launch_cols_fft(g, d, d, dir, COL_PLAIN, nullptr, 1.f, 1, 0);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(data_host, d, NN * sizeof(cpx), cudaMemcpyDeviceToHost));
    cudaFree(d); cudaFree(tw);
    return 0;
    API_CATCH(-1)
}

int fdes_b200_sort_records(unsigned int* keys, int* cols, float* w, int n, int nkeys, int* rowptr,
                           int gpu_index)
{
    API_TRY
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device");
    CK(cudaSetDevice(gpu_index));
    SortBuffers sb{};
    int* rp = nullptr;
    const size_t nn = (size_t)std::max(n, 1);
    CK(cudaMalloc(&sb.keys, nn * 4)); CK(cudaMalloc(&sb.keys_tmp, nn * 4));
    CK(cudaMalloc(&sb.cols, nn * 4)); CK(cudaMalloc(&sb.cols_tmp, nn * 4));
    CK(cudaMalloc(&sb.w, nn * 4)); CK(cudaMalloc(&sb.w_tmp, nn * 4));
    CK(cudaMalloc(&sb.hist, 256 * (size_t)sort_num_blocks(n) * 4));
    CK(cudaMalloc(&rp, ((size_t)nkeys + 1) * 4));
    CK(cudaMemcpy(sb.keys, keys, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(sb.cols, cols, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(sb.w, w, (size_t)n * 4, cudaMemcpyHostToDevice));
    int bits = 0;
    while ((1LL << bits) <= (long long)nkeys) bits++;
    launch_radix_sort(sb, n, bits, 1, 0);
    launch_row_pointers(sb.keys, n, rp, nkeys, 1, 0);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(keys, sb.keys, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cols, sb.cols, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(w, sb.w, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(rowptr, rp, ((size_t)nkeys + 1) * 4, cudaMemcpyDeviceToHost));
    cudaFree(sb.keys); cudaFree(sb.keys_tmp); cudaFree(sb.cols); cudaFree(sb.cols_tmp);
    cudaFree(sb.w); cudaFree(sb.w_tmp); cudaFree(sb.hist); cudaFree(rp);
    return 0;
    API_CATCH(-1)
}

}  // extern "C"

namespace {

// device allocations and the stream of one call, released on every path out of it
struct DeviceAllocs {
    std::vector<void*> p;
    cudaStream_t st = nullptr;
    ~DeviceAllocs()
    {
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
        for (void* q : p) cudaFree(q);
    }
    void* get(size_t bytes)
    {
        void* q = nullptr;
        CK(cudaMalloc(&q, std::max<size_t>(bytes, 4)));
        p.push_back(q);
        return q;
    }
};

// the deposit records of S1 / S2 as the engine lays them out: per configuration nkeys + 1 row pointers,
// then the row masks (launch_row_masks) where the size has them
struct RecordRows {
    int* dev = nullptr;
    size_t stride = 0;
    int mask_off = 0;
};
RecordRows upload_row_pointers(DeviceAllocs& da, const int* rp_host, int nconf, int nkeys, int N, int rec_stride,
                               cudaStream_t st)
{
    for (int c = 0; c < nconf; c++) {
        const int* rp = rp_host + (size_t)c * (nkeys + 1);
        if (rp[0] < 0 || rp[nkeys] > rec_stride) throw std::runtime_error("sweep test: row pointers outside the records");
        for (int k = 0; k < nkeys; k++)
            if (rp[k + 1] < rp[k]) throw std::runtime_error("sweep test: row pointers must not decrease");
    }
    const int E = line_points(N);
    RecordRows r;
    r.stride = (size_t)nkeys + 1 + (E > 0 ? (size_t)(nkeys / N) * (N / E) : 0);
    r.mask_off = E > 0 ? nkeys + 1 : 0;
    r.dev = static_cast<int*>(da.get((size_t)nconf * r.stride * sizeof(int)));
    for (int c = 0; c < nconf; c++)
        CK(cudaMemcpyAsync(r.dev + (size_t)c * r.stride, rp_host + (size_t)c * (nkeys + 1), ((size_t)nkeys + 1) * sizeof(int),
                           cudaMemcpyHostToDevice, st));
    if (E > 0) launch_row_masks(r.dev, r.stride, nkeys, N, E, nconf, st);
    return r;
}

// CTA count of the pipelined column sweeps for the duration of one sweep test; restores the previous value on
// every way out
struct PipeCtasGuard {
    int saved;
    explicit PipeCtasGuard(int ctas) : saved(pipe_cta_cap) { pipe_cta_cap = ctas; pipe_last_grid = 0; }
    ~PipeCtasGuard() { pipe_cta_cap = saved; }
    PipeCtasGuard(const PipeCtasGuard&) = delete;
    PipeCtasGuard& operator=(const PipeCtasGuard&) = delete;
};

}  // namespace

extern "C" {

int fdes_b200_sweep_test(int op, int N, int batch, const int* iargs, int n_iargs, const float* fargs, int n_fargs,
                         float** bufs, const long long* buf_elems, int nbufs, int gpu_index, int pipe_ctas,
                         int* pipe_grid_out)
{
    API_TRY
    if (pipe_grid_out) *pipe_grid_out = 0;
    if (pipe_ctas < 0) throw std::runtime_error("sweep test: pipe_ctas must be >= 0");
    auto ia = [&](int i) {
        if (i >= n_iargs) throw std::runtime_error("sweep test: too few integer arguments");
        return iargs[i];
    };
    auto fa = [&](int i) {
        if (i >= n_fargs) throw std::runtime_error("sweep test: too few float arguments");
        return fargs[i];
    };
    auto need = [&](int i, size_t words) {
        if (i >= nbufs || !bufs[i] || buf_elems[i] < (long long)words)
            throw std::runtime_error("sweep test: buffer " + std::to_string(i) + " needs " + std::to_string(words) + " words");
    };
    // ops from FDES_B200_SCATTER_TABLE on run no sweep: N is any grid size or element count
    const bool sweep = op < FDES_B200_SCATTER_TABLE;
    if (sweep && !fft_size_supported(N)) throw std::runtime_error("unsupported FFT size");
    if (N < 1) throw std::runtime_error("sweep test: N must be >= 1");
    if (op == FDES_B200_SWEEP_GEOM) {
        need(0, 5);
        const SweepGeom g = make_sweep_geom(N, nullptr, 0);
        int* o = reinterpret_cast<int*>(bufs[0]);
        o[0] = g.N; o[1] = g.lo_end; o[2] = g.hi_start; o[3] = line_points(N); o[4] = sweeps_pipelined(N) ? 1 : 0;
        return 0;
    }
    if (batch < 1) throw std::runtime_error("sweep test: batch must be >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device");
    CK(cudaSetDevice(gpu_index));
    const size_t NN = (size_t)N * N, IMG = 2 * NN, Q = (size_t)(N / 2 + 1);
    for (int i = 0; i < nbufs; i++)
        if (buf_elems[i] < 0 || (buf_elems[i] > 0 && !bufs[i])) throw std::runtime_error("sweep test: bad buffer");

    DeviceAllocs da;
    // the sweeps run as in the engine: on a non-blocking stream, launched with programmatic serialisation; every
    // copy of this call is queued on the same stream, so the row masks and the sweep see the uploaded data
    CK(cudaStreamCreateWithFlags(&da.st, cudaStreamNonBlocking));
    const cudaStream_t st = da.st;
    std::vector<cpx> twh;
    SweepGeom g{};
    if (sweep) {
        twh = make_twiddles(N);
        cpx* tw = static_cast<cpx*>(da.get(twh.size() * sizeof(cpx)));
        CK(cudaMemcpyAsync(tw, twh.data(), twh.size() * sizeof(cpx), cudaMemcpyHostToDevice, st));
        g = make_sweep_geom(N, tw, 0);
    }
    // row pointers of S1 / S2 (buffer rp_buf) go up in the engine's layout, not word for word
    int rp_buf = -1, nconf = 0, nkeys = 0;
    RecordRows rows;
    if (op == FDES_B200_SWEEP_DENSITY || op == FDES_B200_SWEEP_POTENTIAL) {
        const int slice = ia(0), slice2 = ia(1), nZ = ia(2), nslices = ia(3), cfg_stride = ia(4), cfg_off2 = ia(5);
        nconf = ia(6);
        const int rec_stride = op == FDES_B200_SWEEP_DENSITY ? ia(7) : INT_MAX;
        if (nZ < 1 || nslices < 1 || slice < 0 || slice >= nslices || slice2 >= nslices || cfg_stride < 1 || cfg_off2 < 0)
            throw std::runtime_error("sweep test: bad slice / species / configuration arguments");
        if ((long long)(batch - 1) * cfg_stride + cfg_off2 >= nconf) throw std::runtime_error("sweep test: too few configurations");
        if ((long long)nslices * nZ * N >= (1LL << 31) - 2) throw std::runtime_error("sweep test: too many row keys");
        nkeys = nslices * nZ * N;
        rp_buf = op == FDES_B200_SWEEP_DENSITY ? 1 : 3;
        need(rp_buf, (size_t)nconf * (nkeys + 1));
        if (op == FDES_B200_SWEEP_DENSITY) {
            need(2, (size_t)nconf * rec_stride); need(3, (size_t)nconf * rec_stride);
            const int* cols = reinterpret_cast<const int*>(bufs[2]);
            for (size_t i = 0; i < (size_t)nconf * rec_stride; i++)
                if (cols[i] < 0 || cols[i] >= N) throw std::runtime_error("sweep test: record column outside the grid");
        }
        rows = upload_row_pointers(da, reinterpret_cast<const int*>(bufs[rp_buf]), nconf, nkeys, N,
                                   op == FDES_B200_SWEEP_DENSITY ? rec_stride : INT_MAX, st);
        g.mask_off = rows.mask_off;
    }
    std::vector<float*> d(nbufs, nullptr);
    for (int i = 0; i < nbufs; i++) {
        if (i == rp_buf || buf_elems[i] == 0) continue;
        d[i] = static_cast<float*>(da.get((size_t)buf_elems[i] * 4));
        CK(cudaMemcpyAsync(d[i], bufs[i], (size_t)buf_elems[i] * 4, cudaMemcpyHostToDevice, st));
    }
    auto c = [&](int i) { return reinterpret_cast<cpx*>(d[i]); };

    const PipeCtasGuard pipe_schedule(pipe_ctas);
    switch (op) {
        case FDES_B200_SWEEP_DENSITY: {
            const int nZ = ia(2);
            need(0, (size_t)batch * nZ * IMG);
            launch_density_rows(g, c(0), rows.dev, reinterpret_cast<const int*>(d[2]), d[3], ia(0), ia(1), nZ, batch,
                                (size_t)ia(7), rows.stride, st, ia(4), ia(5));
        } break;
        case FDES_B200_SWEEP_POTENTIAL: {
            const int nZ = ia(2);
            need(0, (size_t)batch * IMG); need(1, (size_t)batch * nZ * IMG); need(2, (size_t)nZ * Q * Q);
            launch_potential_cols(g, c(0), c(1), d[2], rows.dev, ia(0), ia(1), nZ, batch, rows.stride, st, ia(4), ia(5));
        } break;
        case FDES_B200_SWEEP_TRANSMIT: {
            const int npair = ia(0);
            if (npair < 1 || npair > 2) throw std::runtime_error("sweep test: npair must be 1 or 2");
            need(0, (size_t)batch * IMG); need(1, 2 * (size_t)batch * IMG);
            launch_transmit_rows(g, c(0), c(1), npair, fa(0), batch, st);
        } break;
        case FDES_B200_SWEEP_BANDLIMIT: {
            const int npair = ia(0);
            if (npair < 0 || npair > 2) throw std::runtime_error("sweep test: npair must be 0, 1 or 2");
            need(0, (size_t)(npair ? 2 * batch : batch) * IMG);
            launch_bandlimit_cols(g, c(0), batch, npair, st);
        } break;
        case FDES_B200_SWEEP_MULTIPLY: {
            const int es = ia(0);
            if (es < 0) throw std::runtime_error("sweep test: negative image stride");
            need(0, (size_t)batch * IMG); need(1, ((size_t)(batch - 1) * es + 1) * IMG);
            launch_multiply_rows(g, c(0), c(1), (size_t)es * NN, batch, ia(1) != 0, st);
        } break;
        case FDES_B200_SWEEP_PROPAGATE:
            need(0, (size_t)batch * IMG); need(1, 2 * Q * Q);
            launch_propagate_cols(g, c(0), c(1), batch, st);
            break;
        case FDES_B200_SWEEP_PROPAGATE_FROM: {
            const int stride = ia(0), images = ia(1);
            if (stride < 1 || (long long)(batch - 1) * stride >= images) throw std::runtime_error("sweep test: bad source stack");
            need(0, (size_t)batch * IMG); need(1, (size_t)images * IMG); need(2, 2 * Q * Q);
            const bool lens = nbufs > 3 && buf_elems[3] > 0;
            if (lens) need(3, IMG);
            launch_propagate_cols_from(g, c(0), c(1), stride, images, c(2), batch, ia(2) != 0, lens ? c(3) : nullptr, st);
        } break;
        case FDES_B200_SWEEP_COLS_FFT: {
            const int colop = ia(0);
            const bool in_place = n_iargs > 2 && ia(2) != 0;
            if (colop < COL_PLAIN || colop > COL_DP_ACCUM) throw std::runtime_error("sweep test: unknown column operation");
            if (in_place && colop != COL_PLAIN && colop != COL_MUL_REAL_INV)
                throw std::runtime_error("sweep test: in place only with COL_PLAIN or COL_MUL_REAL_INV");
            need(0, (size_t)batch * IMG);
            if (!in_place) need(1, (size_t)batch * (colop == COL_DP_ACCUM ? NN : IMG));
            if (colop == COL_MUL_CPX_INV) need(2, IMG);
            if (colop == COL_MUL_REAL_INV) need(2, NN);
            launch_cols_fft(g, c(0), in_place ? d[0] : d[1], ia(1), (ColOp)colop, nbufs > 2 ? d[2] : nullptr, fa(0), batch, st);
        } break;
        case FDES_B200_SWEEP_ROWS_FFT_SUM: {
            const int epi = ia(0);
            if (epi != ROW_ACCUM && epi != ROW_INTENS_ACCUM) throw std::runtime_error("sweep test: ROW_ACCUM or ROW_INTENS_ACCUM");
            need(0, (size_t)batch * IMG); need(1, epi == ROW_ACCUM ? IMG : NN);
            RowOpts ro;
            ro.scale = fa(0);
            ro.band_only_in = ia(1) != 0;
            launch_rows_fft_sum(g, c(0), d[1], +1, (RowEpilogue)epi, ro, batch, st);
        } break;
        case FDES_B200_SWEEP_ROWS_FFT: {
            const int dir = ia(0), epi = ia(1);
            RowOpts ro;
            ro.scale = fa(0);
            ro.in_is_real = ia(2) != 0;
            ro.band_only_in = ia(3) != 0;
            ro.band_only_out = ia(4) != 0;
            ro.dn1 = ia(5); ro.dn2 = ia(6); ro.n1 = ia(7); ro.n2 = ia(8);
            const bool in_place = ia(9) != 0;
            if (dir != -1 && dir != 1) throw std::runtime_error("sweep test: dir must be -1 or +1");
            if (epi < ROW_STORE || epi > ROW_CROP_REAL) throw std::runtime_error("sweep test: unknown row epilogue");
            if (ro.band_only_out && epi != ROW_STORE) throw std::runtime_error("sweep test: band_only_out only with ROW_STORE");
            if (in_place && (epi != ROW_STORE || ro.in_is_real))
                throw std::runtime_error("sweep test: in place only with ROW_STORE and complex input");
            if (epi == ROW_CROP_REAL && (ro.n1 < 1 || ro.n2 < 1 || ro.dn1 < 0 || ro.dn2 < 0 || ro.dn1 > N - ro.n1 || ro.dn2 > N - ro.n2))
                throw std::runtime_error("sweep test: crop window outside the grid");
            need(0, (size_t)batch * (ro.in_is_real ? NN : IMG));
            if (!in_place)
                need(1, (size_t)batch * (epi == ROW_INTENS_ACCUM ? NN : epi == ROW_CROP_REAL ? (size_t)ro.n1 * ro.n2 : IMG));
            launch_rows_fft(g, d[0], in_place ? d[0] : d[1], dir, (RowEpilogue)epi, ro, batch, st);
        } break;
        case FDES_B200_SWEEP_PROBE:
            need(0, (size_t)batch * IMG); need(1, IMG); need(2, 2 * (size_t)batch);
            launch_probe_cols(g, c(0), c(1), d[2], batch, st);
            break;
        case FDES_B200_SWEEP_DETECTOR: {
            DetectorRings rings{};
            rings.n = ia(0);
            if (rings.n < 1 || rings.n > MAX_DETECTORS) throw std::runtime_error("sweep test: 1.." + std::to_string(MAX_DETECTORS) + " detectors");
            for (int r = 0; r < rings.n; r++) { rings.in2[r] = fa(3 + r); rings.out2[r] = fa(3 + rings.n + r); }
            need(0, (size_t)batch * IMG); need(1, (size_t)batch * rings.n);
            // a tile the detector sweep leaves unwritten reaches `out` as NaN
            const size_t np = (size_t)batch * detector_tiles(g) * MAX_DETECTORS;
            float* partial = static_cast<float*>(da.get(np * sizeof(float)));
            launch_fill_f32(partial, np, std::nanf(""), st);
            launch_detector_cols(g, c(0), partial, d[1], rings, fa(0), fa(1), fa(2), batch, st);
        } break;
        case FDES_B200_SWEEP_DETECTOR4D: {
            const int Q = ia(0), bin = ia(1);
            if (Q < 1) throw std::runtime_error("sweep test: window must be >= 1");
            stem4d_window(N, Q, bin);
            const size_t S = (size_t)(Q / bin);
            need(0, (size_t)batch * IMG); need(1, (size_t)batch * S * S);
            // scratch: NaN in the band columns (the sweep must write each of their window pixels before the bins are
            // summed), 0 in the others (the engine zeroes them once per scan)
            std::vector<float> h((size_t)batch * Q * Q);
            for (size_t i = 0; i < h.size(); i++) {
                const int kx = (int)((i % Q) + (N - Q) / 2 + N - N / 2) % N;
                h[i] = (kx < g.lo_end || kx >= g.hi_start) ? std::nanf("") : 0.f;
            }
            float* scratch = static_cast<float*>(da.get(h.size() * sizeof(float)));
            CK(cudaMemcpyAsync(scratch, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, st));
            launch_detector4d_cols(g, c(0), scratch, d[1], Q, bin, fa(0), batch, st);
            CK(cudaStreamSynchronize(st));     // h goes out of scope
        } break;
        case FDES_B200_SCATTER_TABLE:
            need(0, Q * Q);
            launch_scattering_table(d[0], N, kirkland_row(ia(0)), fa(0), fa(1), fa(2), Params().cst_pi, st);
            break;
        case FDES_B200_PROP_TABLE:
            need(0, 2 * Q * Q);
            launch_propagator_table(c(0), N, fa(0), fa(1), fa(2), fa(3), Params().cst_pi, st);
            break;
        case FDES_B200_LENS_TABLE: {
            need(0, IMG);
            LensParams lp;
            for (int a = 0; a < AB_COUNT; a++) { lp.ab0[a] = fa(a); lp.ab1[a] = fa(AB_COUNT + a); }
            lp.defocus_k = fa(28); lp.defocspread = fa(29); lp.lambda = fa(30); lp.d1 = fa(31); lp.d2 = fa(32);
            lp.ObjAp = fa(33); lp.pi = Params().cst_pi; lp.mode = ia(0);
            launch_lens_table(c(0), N, lp, fa(34), st, ia(1) != 0);
        } break;
        case FDES_B200_DETECTOR_TABLE: {
            need(0, NN);
            DetectorParams dp;
            dp.mtfa = fa(0); dp.mtfb = fa(1); dp.mtfc = fa(2); dp.mtfd = fa(3); dp.illangle = fa(4); dp.defocus_k = fa(5);
            dp.lambda = fa(6); dp.d1 = fa(7); dp.d2 = fa(8); dp.pi = Params().cst_pi;
            dp.mode = ia(0); dp.use_incoherence = ia(1); dp.use_mtf = ia(2);
            launch_detector_table(d[0], N, dp, fa(9), st);
        } break;
        case FDES_B200_TILT_BEAM:
            if (ia(0) != 1 && ia(0) != -1) throw std::runtime_error("sweep test: flag must be +1 or -1");
            need(0, IMG);
            launch_tilt_beam(c(0), N, fa(0), fa(1), fa(2), fa(3), fa(4), Params().cst_pi, ia(0), st);
            break;
        case FDES_B200_TUKEY:
        case FDES_B200_AREA_MASK:
            if (ia(0) < 0 || ia(0) > N || ia(1) < 0 || ia(1) > N) throw std::runtime_error("sweep test: dn1, dn2 must be in [0, N]");
            need(0, IMG);
            if (op == FDES_B200_TUKEY) launch_tukey_window(c(0), N, ia(0), ia(1), Params().cst_pi, st);
            else launch_area_mask_blend(c(0), N, ia(0), ia(1), st);
            break;
        case FDES_B200_NORM2: {
            need(0, 2 * (size_t)N); need(1, 2);
            double* dd = static_cast<double*>(da.get(257 * sizeof(double)));
            launch_norm2(c(0), (size_t)N, dd, dd + 256, st);
            CK(cudaMemcpyAsync(d[1], dd + 256, sizeof(double), cudaMemcpyDeviceToDevice, st));
        } break;
        case FDES_B200_PEER_SUM: {
            PeerSources src{};
            src.n = ia(0);
            if (src.n < 1 || src.n > MAX_PEERS) throw std::runtime_error("sweep test: 1.." + std::to_string(MAX_PEERS) + " sources");
            for (int r = 0; r <= src.n; r++) need(r, (size_t)N);
            for (int r = 0; r < src.n; r++) src.p[r] = d[1 + r];
            launch_peer_sum(d[0], src, (size_t)N, st);
        } break;
        case FDES_B200_JITTER: {
            const size_t n3 = 3 * (size_t)N;
            if (n_iargs < 2 || n_iargs % 2) throw std::runtime_error("sweep test: (burn, nconf) pairs expected");
            long long confs = 0;
            for (int i = 0; i < n_iargs; i += 2) {
                if (ia(i) >= 0 && ia(i + 1) < 1) throw std::runtime_error("sweep test: nconf must be >= 1");
                if (ia(i) >= 0) confs += ia(i + 1);
            }
            if (n3 > INT_MAX) throw std::runtime_error("sweep test: too many atoms");
            need(0, n3); need(1, (size_t)N); need(2, (size_t)confs * n3);
            void* states = da.get(rng_state_bytes() * n3);
            launch_rng_init(states, (int)n3, 1ULL, st);
            float* out = d[2];
            for (int i = 0; i < n_iargs; i += 2) {
                if (ia(i) < 0) { launch_rng_init(states, (int)n3, 1ULL, st); continue; }   // the streams start again
                launch_atom_jitter(out, d[0], d[1], N, states, ia(i), ia(i + 1), st);
                out += (size_t)ia(i + 1) * n3;
            }
        } break;
        case FDES_B200_ANSCOMBE: {
            const bool second = nbufs > 1 && buf_elems[1] > 0;
            need(0, 2 * (size_t)N);
            if (second) need(1, 2 * (size_t)N);
            void* states = da.get(rng_state_bytes() * (size_t)N);
            launch_rng_init(states, N, (unsigned long long)ia(0), st);
            launch_anscombe_noise(c(0), (size_t)N, fa(0), states, st);
            if (second) launch_anscombe_noise(c(1), (size_t)N, fa(0), states, st);
        } break;
        case FDES_B200_PLANE_WAVE:
            need(0, (size_t)batch * IMG);
            launch_plane_wave_rowspace(c(0), N, batch, st);
            break;
        case FDES_B200_ZERO_OUTBAND:
            if (ia(0) < 0 || ia(1) < ia(0) || ia(1) > N) throw std::runtime_error("sweep test: need 0 <= lo_end <= hi_start <= N");
            need(0, (size_t)batch * IMG);
            launch_zero_outband(c(0), N, ia(0), ia(1), batch, st);
            break;
        case FDES_B200_ABSORPTIVE:
            need(0, 2 * (size_t)N);
            launch_absorptive_factor(c(0), (size_t)N, fa(0), st);
            break;
        case FDES_B200_SCALE_CPX:
            need(0, 2 * (size_t)N);
            launch_scale_cpx(c(0), (size_t)N, fa(0), st);
            break;
        case FDES_B200_RECORDS: {
            const int m3 = ia(0), nZ = ia(1), nconf_r = ia(2);
            const int nAt = nbufs > 1 ? (int)std::min<long long>(buf_elems[1], INT_MAX / 4) : 0;
            if (m3 < 1 || nZ < 1 || nconf_r < 1 || nAt < 1) throw std::runtime_error("sweep test: bad records arguments");
            if ((long long)m3 * nZ * N >= (1LL << 31) - 2) throw std::runtime_error("sweep test: too many row keys");
            const int nk = m3 * nZ * N, nrec = 4 * nAt;
            int key_bits = 0;
            while ((1LL << key_bits) <= (long long)nk) key_bits++;
            const int E = fft_size_supported(N) ? line_points(N) : 0;
            const size_t rp_stride = (size_t)nk + 1 + (E > 0 ? (size_t)(nk / N) * (N / E) : 0);
            const size_t nr = (size_t)nconf_r * nrec;
            need(0, (size_t)nconf_r * 3 * nAt); need(2, nAt); need(3, nr); need(4, nr); need(5, nr);
            need(6, (size_t)nconf_r * rp_stride);
            const int* zi = reinterpret_cast<const int*>(bufs[1]);
            for (int i = 0; i < nAt; i++)
                if (zi[i] < 0 || zi[i] >= nZ) throw std::runtime_error("sweep test: species index outside [0, nZ)");
            SortBuffers sb{reinterpret_cast<uint32_t*>(d[3]), static_cast<uint32_t*>(da.get(nr * 4)),
                           reinterpret_cast<int*>(d[4]), static_cast<int*>(da.get(nr * 4)), d[5],
                           static_cast<float*>(da.get(nr * 4)),
                           static_cast<unsigned int*>(da.get((size_t)nconf_r * 256 * sort_num_blocks(nrec) * 4))};
            const BinGeom bg{N, N, m3, nZ, fa(0), fa(1), fa(2)};
            launch_build_records(d[0], reinterpret_cast<const int*>(d[1]), d[2], nAt, bg, sb, reinterpret_cast<int*>(d[6]),
                                 rp_stride, key_bits, E, nconf_r, st);
        } break;
        default: throw std::runtime_error("sweep test: unknown op " + std::to_string(op));
    }
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < nbufs; i++) {
        if (i == rp_buf) {
            for (int cf = 0; cf < nconf; cf++)
                CK(cudaMemcpyAsync(bufs[i] + (size_t)cf * (nkeys + 1), rows.dev + (size_t)cf * rows.stride,
                                   ((size_t)nkeys + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
        } else if (buf_elems[i] > 0) {
            CK(cudaMemcpyAsync(bufs[i], d[i], (size_t)buf_elems[i] * 4, cudaMemcpyDeviceToHost, st));
        }
    }
    CK(cudaStreamSynchronize(st));
    if (pipe_grid_out) *pipe_grid_out = pipe_last_grid;
    return 0;
    API_CATCH(-1)
}

}  // extern "C"

// "<count>" -> first, first + 1, ... (modulo the device count); "<i>,<j>,..." -> that list;
// empty / NULL -> {first}
std::vector<int> fdes_b200_gpu_list(const char* spec, int first)
{
    std::vector<int> out;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess) ndev = 0;
    if (!spec || !spec[0]) { out.push_back(first); return out; }
    if (strchr(spec, ',')) {
        const char* q = spec;
        while (*q) {
            char* end = nullptr;
            const long v = strtol(q, &end, 10);
            if (end == q) break;
            out.push_back((int)v);
            q = *end == ',' ? end + 1 : end;
        }
    } else {
        int n = atoi(spec);
        if (ndev > 0 && n > ndev) n = ndev;
        for (int i = 0; i < std::max(1, n); i++) out.push_back(ndev > 0 ? (first + i) % ndev : first + i);
    }
    if (out.empty()) out.push_back(first);
    return out;
}

extern "C" {

int fdes_b200_parse_gpu_list(const char* spec, int first, int* out, int max_out)
{
    const std::vector<int> v = fdes_b200_gpu_list(spec, first);
    for (int i = 0; i < (int)v.size() && i < max_out; i++) out[i] = v[i];
    return (int)v.size();
}

// ---------------------------------------------------------------------------------------------
// drop-in export (reference src/FDESExport.cu:59-178)
// ---------------------------------------------------------------------------------------------
void FDES(int gpu_Index, int print_Level, char* input_name, char* image_name, char* emd_save_name,
          float* atomsArray, int numAtoms, float* dstImage)
{
    fprintf(stderr, "\n  fdes_b200: B200-native forward multislice behind the FDES interface\n\n");
    fprintf(stderr, "   input_name %s  \n", input_name ? input_name : "(null)");
    if (!input_name || !(strstr(input_name, ".emd") || strstr(input_name, ".cnf") || strstr(input_name, ".qsc"))) {
        fprintf(stderr, " \n input file %s error   \n", input_name ? input_name : "(null)");
        exit(0);   // reference: src/FDESExport.cu:100-101
    }
    if (numAtoms <= 0) exit(0);   // readAtomsFromArray, src/paramStructure.cu:306-307
    if (print_Level < 0 || print_Level > 2) {
        fprintf(stderr, " \n printLevel error %s  \n", input_name);
        exit(EXIT_FAILURE);
    }
    using clk = std::chrono::steady_clock;
    const bool timing = getenv("FDES_B200_TIMING") != nullptr;
    const auto t0 = clk::now();
    // FDES_B200_GPUS = "<count>" (devices gpu_Index, gpu_Index + 1, ...) or "<i>,<j>,..." shards the
    // run over several GPUs of this process; unset: the reference's single device (gpu_Index)
    const std::vector<int> gpus = fdes_b200_gpu_list(getenv("FDES_B200_GPUS"), gpu_Index);
    fdes_b200_sim* sim = gpus.size() > 1
        ? fdes_b200_open_multi(input_name, atomsArray, numAtoms, gpus.data(), (int)gpus.size(), 0, print_Level > 1)
        : fdes_b200_open_cnf(input_name, atomsArray, numAtoms, gpus.empty() ? gpu_Index : gpus[0], 0, 0, 1, print_Level > 1);
    if (!sim) {
        fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error());
        exit(EXIT_FAILURE);
    }
    const auto t1 = clk::now();
    // side-effect file of getParams (src/paramStructure.cu:629-631), written by a helper thread
    // while the GPU works (formatting tens of thousands of atom lines takes milliseconds)
    // (readQsc writes ParamsUsedQsc.txt instead, src/rwQsc.cu:1084)
    // (readQsc writes ParamsUsedQsc.txt, readHdf5 ParamsUsedEmd.txt instead: src/rwQsc.cu:1084,
    // src/rwHdf5.cu:2565); .cnf and .qsc inputs also leave "config.emd" behind (src/FDESExport.cu:123, 141)
    const bool from_emd = strstr(input_name, ".emd") != nullptr;
    const char* used_name = from_emd ? "ParamsUsedEmd.txt"
                          : (is_qsc_name(input_name) && !strstr(input_name, ".cnf")) ? "ParamsUsedQsc.txt" : "dataFDES_used.cnf";
    std::thread cnf_writer([sim, gpu_Index, used_name, from_emd] {
        write_cnf(used_name, sim->params, sim->atoms, gpu_Index);
        if (!from_emd) write_emd("config.emd", sim->params, sim->atoms, nullptr, nullptr, 0, nullptr);
    });
    fprintf(stderr, "  Number of atoms %d \n", sim->atoms.size());
    const Params& p = sim->eng->params();
    const size_t n123 = (size_t)p.n1 * p.n2 * p.n3, m12 = (size_t)p.m1 * p.m2;
    // the caller's buffer receives the images directly (exportFormedimage, src/FDESExport.cu:162)
    std::vector<float> image_own, ew, pot;
    float* image = dstImage;
    if (!image) { image_own.resize(n123); image = image_own.data(); }
    if (print_Level > 1) ew.resize(2 * m12 * p.n3);
    auto fail = [&](void) {
        fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error());
        cnf_writer.join();
        exit(EXIT_FAILURE);
    };
    if (fdes_b200_simulate(sim, image, ew.empty() ? nullptr : ew.data()) != 0) fail();
    const auto t2 = clk::now();
    if (print_Level > 0) {
        pot.resize(2 * m12 * (size_t)sim->m3_orig);
        if (fdes_b200_potential(sim, pot.data()) != 0) fail();
    }
    {
        // results file of buildMeasurements (src/crystalMaker.cu:402 -> writeHdf5, src/rwHdf5.cu:27-1084):
        // HDF5 bytes written by our own serialiser (emd.cpp; no libhdf5 in this build), on a helper
        // thread while this one writes the raw image file
        std::thread emd_writer;
        if (emd_save_name && emd_save_name[0])
            emd_writer = std::thread([&] {
                write_emd(emd_save_name, sim->params, sim->atoms, image, pot.empty() ? nullptr : pot.data(),
                          sim->m3_orig, ew.empty() ? nullptr : ew.data());
            });
        if (image_name && image_name[0]) write_binary(image_name, image, n123);
        if (emd_writer.joinable()) emd_writer.join();
    }
    const auto t3 = clk::now();
    cnf_writer.join();
    fdes_b200_close(sim);
    const auto t4 = clk::now();
    if (timing) {
        auto ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "  fdes_b200 timing [ms]: open %.2f  simulate %.2f  outputs %.2f  close %.2f  total %.2f\n",
                ms(t0, t1), ms(t1, t2), ms(t2, t3), ms(t3, t4), ms(t0, t4));
    }
}

void fdes_b200_release_cache(void) { release_device_cache(); }

}  // extern "C"
