/* fdes_b200 -- C ABI of the B200-native FDES forward-multislice library (libfdes_b200.so).
 *
 * Plain C: pointers and sizes only, no C++ or torch types.  Two layers:
 *
 *  (1) The drop-in symbol.  `FDES` has the exact signature the reference exports from
 *      libFDES_SHARED_LIB.so (reference src/FDESExport.cu:59-60) and that
 *      Python/pyFDES.py:33-41 binds through ctypes, so `ctypes.CDLL("libfdes_b200.so").FDES`
 *      (or a symlink named libFDES_SHARED_LIB.so) replaces it without touching the caller.
 *
 *  (2) A session API over the same engine.  It exposes the seam the reference keeps internal
 *      (buildMeasurements, include/crystalMaker.h:77) so a host framework can shard frozen-phonon
 *      configurations over several GPUs (one process per GPU) and reduce the partial intensity /
 *      exit-wave sums itself (e.g. torch.distributed all_reduce over NCCL), plus the building
 *      blocks the parity tests compare against the oracle.
 *
 * All functions returning int return 0 on success and -1 on failure; the message is available
 * from fdes_b200_last_error().  There is no CPU fallback: without a CUDA device every entry point
 * that computes fails.
 */
#ifndef FDES_B200_H
#define FDES_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- (1) drop-in for the reference export ------------------------------------------------
 * Replaces: extern "C" void FDES(...)                     reference src/FDESExport.cu:59-178
 *   gpu_Index      CUDA device ordinal                    (:68, :106)
 *   print_Level    0 images | 1 + potential | 2 + exit waves (:69)
 *   input_name     parameter file: ".emd", ".cnf" or ".qsc", tested in that order     (:73-102)
 *   image_name     raw float32 output file [n3][n2][n1]    (src/crystalMaker.cu:399)
 *   emd_save_name  results file, EMD/HDF5 with the reference's groups (src/rwHdf5.cu:27-1084)
 *   atomsArray     host float32 [numAtoms][6] = Z, x, y, z [m], DWF [m^2], occupancy
 *                                                          (src/paramStructure.cu:316-324)
 *   dstImage       host float32 [n3][n2][n1], caller-allocated (:162, src/paramStructure.cu:347-359)
 * Like the reference it returns void and terminates the process (exit) on unusable input. */
void FDES(int gpu_Index, int print_Level, char* input_name, char* image_name, char* emd_save_name,
          float* atomsArray, int numAtoms, float* dstImage);

/* ---- (2) session API ---------------------------------------------------------------------- */
typedef struct fdes_b200_sim fdes_b200_sim;

const char* fdes_b200_last_error(void);
/* Device memory blocks are cached per process between simulations (FDES() calls included) so that
 * repeated calls do not pay cudaMalloc/cudaFree; this returns the idle ones to the driver. */
void fdes_b200_release_cache(void);
int fdes_b200_version(void);

/* Host-only (no CUDA call): parse a .cnf (or .qsc / .emd) exactly as fdes_b200_open_cnf does and report what the
 * engine would run (readConfig + consitentParams, src/paramStructure.cu:42-302, 637-673; sub-slice
 * logic src/crystalMaker.cu:720-743).  dims[10] = n1 n2 n3 m1 m2 m3(after sub-slicing) nAt nZ
 * frozen_phonons mode; scalars[8] as fdes_b200_get_scalars; per_k [n3][5] = specimen_tilt x y,
 * beam_tilt x y, defocus (may be NULL); atoms6_out [max_atoms][6] (may be NULL).
 * Returns the number of atoms in the file, -1 on failure. */
int fdes_b200_parse_cnf(const char* cnf_path, int* dims, float* scalars, float* per_k,
                        float* atoms6_out, int max_atoms);

/* Host-only (no CUDA call): read a .cnf / .qsc / .emd parameter file exactly as fdes_b200_open_cnf does and
 * write parameters + atoms back in .cnf syntax -- the side-effect file the reference leaves behind
 * (writeConfig, src/paramStructure.cu:360-487: "dataFDES_used.cnf" from getParams :629-631,
 * "ParamsUsedQsc.txt" from readQsc, src/rwQsc.cu:1084). */
int fdes_b200_write_used_cnf(const char* input_path, const char* out_path);

/* Host-only (no CUDA call): write an EMD (HDF5) file with the reference's layout (writeHdf5,
 * src/rwHdf5.cu:27-1084; the bytes are produced by the library's own serialiser, there is no libhdf5
 * here) from the parameters + atoms of input_path (.cnf / .qsc / .emd) and the caller's arrays:
 * image_host [n3][n2][n1] -> /data/images/data [n1][n2][n3]; potential_host [pot_slices][m2][m1][2]
 * -> /data/potential_slices/data [m1][m2][pot_slices][2]; exitwave_host [n3][m2][m1][2] ->
 * /data/exit_wave/data [m1][m2][n3][2].  Any array may be NULL (all NULL = the "config.emd" of the
 * 6-argument writeHdf5, :1085-1945).  FDES() writes emd_save_name through the same code. */
int fdes_b200_write_emd(const char* input_path, const char* emd_path, const float* image_host,
                        const float* potential_host, int pot_slices, const float* exitwave_host);

/* Open a simulation from a parameter file, selected by name like src/FDESExport.cu:85-102:
 * .emd (readHdf5, src/rwHdf5.cu:1946-2571, parsed by the library's own HDF5 reader),
 * .cnf (reader: getParams, reference src/paramStructure.cu:588-635) or QSTEM .qsc + the .cfg unit
 * cell it names (readQsc, src/rwQsc.cu:8-1088; fdes_b200/csrc/qsc.cpp lists what is refused).
 * atoms6 == NULL: atoms come from the file's `atom:` lines; otherwise [numAtoms][6] like FDES().
 * batch: phonon configurations advanced together (0 = automatic).
 * rank/world: this process handles configurations [count*rank/world, count*(rank+1)/world).
 * want_exitwave: keep the coherent exit-wave average (reference print_level 2). */
fdes_b200_sim* fdes_b200_open_cnf(const char* cnf_path, const float* atoms6, int numAtoms,
                                  int gpu_index, int batch, int rank, int world, int want_exitwave);
/* The same session on `ngpus` devices of THIS process (one engine and, while they compute, one host
 * thread per device) -- the multi-GPU form of the seam below buildMeasurements
 * (include/crystalMaker.h:77; the reference itself is single-GPU, cudaSetDevice at src/FDES.cu:165).
 * What is sharded follows the reference's loop nest (src/crystalMaker.cu:324-372): with frozen phonons
 * the configurations j of every measurement k (contiguous blocks per device, identical RNG streams +
 * burn-in, partial intensities / exit waves summed onto gpu_indices[0] by a kernel that reads the
 * peers' buffers over NVLink, detector tail once per k); without them the measurements k of a tilt /
 * defocus series, or the probe positions of fdes_b200_stem_scan.  fdes_b200_simulate,
 * fdes_b200_stem_scan and fdes_b200_close work on such a session unchanged; the building blocks further down act on
 * the engine of gpu_indices[0].  FDES() opens its session this way when the environment variable
 * FDES_B200_GPUS is set ("4" = gpu_Index .. gpu_Index + 3, or a list "0,2,5"); the CLI has --gpus. */
fdes_b200_sim* fdes_b200_open_multi(const char* cnf_path, const float* atoms6, int numAtoms,
                                    const int* gpu_indices, int ngpus, int batch, int want_exitwave);
/* engines (GPUs) the session actually uses: min(ngpus, independent units) */
int fdes_b200_num_gpus(const fdes_b200_sim* sim);
/* the FDES_B200_GPUS / --gpus syntax -> device ordinals; returns how many (out may be NULL when max_out = 0) */
int fdes_b200_parse_gpu_list(const char* spec, int first, int* out, int max_out);
void fdes_b200_close(fdes_b200_sim* sim);

/* dims[10] = n1 n2 n3 m1 m2 m3(after sub-slicing) nAt nZ phonon_configs batch */
int fdes_b200_get_dims(const fdes_b200_sim* sim, int* dims);
/* scalars[8] = lambda sigma gamma d1 d2 d3(after sub-slicing) E0 imPot */
int fdes_b200_get_scalars(const fdes_b200_sim* sim, float* scalars);

/* Device accumulators for the partial sums of this rank (float32 on the sim's device):
 * intensity_dev [m2*m1], exitwave_dev [m2*m1*2] (may be NULL).  NULL restores the internal ones. */
int fdes_b200_set_accumulators(fdes_b200_sim* sim, float* intensity_dev, float* exitwave_dev);
/* All phonon configurations of this rank for measurement k (loop body of
 * src/crystalMaker.cu:324-367): accumulators <- sum_j (.)/count. */
int fdes_b200_run_k(fdes_b200_sim* sim, int k);
/* Detector tail on the (reduced) accumulators (addNoiseAndMtf, src/crystalMaker.cu:579-613):
 * image_host [n2*n1]; exitwave_host [m2*m1*2] or NULL. */
int fdes_b200_finish_k(fdes_b200_sim* sim, int k, float* image_host, float* exitwave_host);
/* Whole single-GPU run: image_host [n3][n2][n1], exitwave_host [n3][m2][m1][2] or NULL.
 * Host buffers in, host buffers out (this is what FDES() calls). */
int fdes_b200_simulate(fdes_b200_sim* sim, float* image_host, float* exitwave_host);
/* Untilted phonon-free potential slices, original slicing: out_host [m3_orig][m2][m1][2]
 * (src/crystalMaker.cu:381-397).  m3_orig is returned by fdes_b200_potential_slices_count. */
int fdes_b200_potential_slices_count(const fdes_b200_sim* sim);
int fdes_b200_potential(fdes_b200_sim* sim, float* out_host);

/* ---- STEM probe scan (extension; FDES has mode 2 = one CBED probe at the grid centre only,
 * src/multisliceSimulation.cu:572-581, and rejects mode: STEM inputs, src/rwQsc.cu:33-44) --------
 * The .cnf must select mode 2.  A scan position is the reference's probe shifted periodically to
 * xy_host[i] = (x, y) [m] relative to the grid centre; the specimen stays fixed.  Detector d
 * integrates the diffraction intensity |FFT2 psi|^2 / N^2 (diffractionPattern,
 * src/crystalMaker.cu:700-718) over k_in^2 <= |k|^2 < k_out^2 with k = sin(theta * 1e-3) / lambda,
 * theta = det_mrad_host[d] = (inner, outer) [mrad] (detector convention of src/rwQsc.cu:723-730).
 * out_host [nprobes][ndet], averaged over the frozen-phonon configurations; an empty specimen
 * gives n1*n2 on a detector that covers the whole pattern.  Returns the CUDA-event milliseconds
 * of the scan (negative on failure). */
double fdes_b200_stem_scan(fdes_b200_sim* sim, int k, int nprobes, const float* xy_host, int ndet,
                           const float* det_mrad_host, float* out_host);

/* 4D-STEM scan (extension): the diffraction pattern of every probe position instead of ring sums.  Positions,
 * units and frame as fdes_b200_stem_scan.  Pattern p is I_p = |FFT2 psi_p|^2 / N^2 (diffractionPattern,
 * src/crystalMaker.cu:700-718) averaged over the frozen-phonon configurations with weight 1/count, in the
 * reference's fftshift frame (out[(i + N/2) mod N] = in[i]), cropped to the centred window [o, o + Q)^2 with
 * o = (N - Q) / 2 and binned bin x bin by summation: patterns_host [nprobes][Q/bin][Q/bin] float32, qx fastest;
 * window pixel (qy, qx) holds the frequency (qx - Q/2, qy - Q/2) (integer division), the zero frequency sits at
 * [Q/2][Q/2] before binning.  window: Q, with Q = N (mod 2), bin dividing Q and 1 <= Q <= N; 0 = the smallest such Q
 * that holds every frequency the 2/3 band limit keeps (nothing of the pattern is lost, an empty specimen sums to
 * n1*n2).  fdes_b200_stem_4d_side gives Q/bin.
 * ndet (0..8) annular detectors as in fdes_b200_stem_scan run in the same pass: det_out_host [nprobes][ndet],
 * bitwise the signals fdes_b200_stem_scan returns (NULL allowed when ndet = 0).
 * The raster runs in passes of probes_per_pass probes (0 = automatic: the two device pass buffers take at most
 * about a quarter of the free device memory); a finished pass is copied to patterns_host while the next one
 * computes.  Results do not depend on the pass size, the batch size or the number of GPUs the probes are dealt
 * out to; with frozen-phonon configurations sharded over GPUs the passes of the devices are summed on the host in
 * device order.  Returns the CUDA-event milliseconds of the device loop (negative on failure). */
double fdes_b200_stem_scan_4d(fdes_b200_sim* sim, int k, int nprobes, const float* xy_host, int window, int bin, int ndet,
                              const float* det_mrad_host, int probes_per_pass, float* patterns_host, float* det_out_host);
/* Host-only (no CUDA call): the side Q/bin of the 4D-STEM patterns on an N x N grid for window / bin as
 * fdes_b200_stem_scan_4d takes them, -1 with the reason in fdes_b200_last_error() when they are not admissible. */
int fdes_b200_stem_4d_side(int N, int window, int bin);

/* Host-only: the scan raster and detectors a QSTEM `mode: STEM` .qsc describes -- the keys readQsc
 * parses (scan_x_start/stop/pixels, scan_y_*, src/rwQsc.cu:444-466; `detector: inner outer name ..`
 * [mrad], :698-735) but FDES never uses -- in the form fdes_b200_stem_scan takes: nxy[2] = pixels in
 * x, y; xy_host [nx][ny][2] probe positions [m] (QSTEM raster start + i (stop - start) / pixels, moved
 * into the frame of the atoms as readQsc centres them); det_mrad_host [ndet][2].  Returns the number
 * of detectors, -1 on failure.  Call once with NULL arrays to size them. */
int fdes_b200_qsc_scan(const char* qsc_path, int* nxy, float* xy_host, int max_probes, float* det_mrad_host,
                       int max_det);

/* ---- building blocks (parity tests, benchmarks) ------------------------------------------- */
/* next frozen-phonon coordinates for measurement k -> xyz_host [nAt][3]
 * (atomJitter_d, src/crystalMaker.cu:37-48; advances the XORWOW streams) */
int fdes_b200_jitter_next(fdes_b200_sim* sim, int k, float* xyz_host);
/* integer bin tuples (i1, i2, i3, species index) per atom, -1 when the atom is rejected
 * (squareAtoms_d index arithmetic, src/crystalMaker.cu:85-92): bins_host [nAt][4] */
int fdes_b200_bin_atoms(fdes_b200_sim* sim, const float* xyz_host, int* bins_host);
/* phase grating of one slice (phaseGrating, src/crystalMaker.cu:507-536): V_host [m2*m1*2] */
int fdes_b200_phase_grating(fdes_b200_sim* sim, const float* xyz_host, int slice, float* V_host);
/* exit wave of one configuration with given coordinates (incomingWave + m3 x
 * (phaseGrating + forwardPropagation)): psi_host [m2*m1*2] */
int fdes_b200_exit_wave(fdes_b200_sim* sim, const float* xyz_host, int k, float* psi_host);
/* Throughput loop: `configs` configurations with everything resident in HBM; returns the
 * CUDA-event milliseconds of the loop (negative on failure). */
double fdes_b200_bench_configs(fdes_b200_sim* sim, int k, int configs);
/* Average launch duration [ms] of each of the six per-slice sweeps (S1 density rows, S2 potential
 * columns, S3 transmission rows, S4 band-limit columns, S5 multiply rows, S6 propagate columns)
 * over `reps` back-to-back launches on a prepared batch -- the live kernel times behind the
 * roofline figures of bench.py. */
int fdes_b200_time_sweeps(fdes_b200_sim* sim, int k, int batch, int reps, float* ms6);
/* counters[4] = slices executed, kernels launched (since open or last reset), band columns
 * (columns kept by the 2/3 limit, rounded to tiles), 0 */
int fdes_b200_get_counters(fdes_b200_sim* sim, long long* counters, int reset);
/* 2-D complex64 FFT of a host array [N][N] in place with the library's own sweeps
 * (dir -1 forward, +1 unnormalised inverse) -- replaces cufftExecC2C for the tests. */
int fdes_b200_fft2d(float* data_host, int N, int dir, int gpu_index);
/* stable radix sort + row pointers on host arrays (test hook for the binning pipeline):
 * keys [n] (values < nkeys are valid), cols [n], w [n] sorted in place; rowptr [nkeys+1]. */
int fdes_b200_sort_records(unsigned int* keys, int* cols, float* w, int n, int nkeys, int* rowptr,
                           int gpu_index);
/* One sweep of the slice loop, launched once on host arrays (test hook for per-sweep models).
 * bufs[i] holds buf_elems[i] 32-bit words (float, int where noted; a complex image is N*N interleaved
 * float pairs).  Every buffer is uploaded, the sweep runs on the N x N grid with the geometry the
 * engine uses (band columns, row masks of the deposit records), and every buffer is downloaded again,
 * so that what a sweep must not write still holds what the caller put there.  -1 on failure (also
 * when a buffer is too small for the arguments, or the size has no such sweep).
 * pipe_ctas: CTAs of the pipelined column sweeps (persistent CTAs that walk tiles t, t + grid, ...):
 * 0 = as in the engine, one per SM; c >= 1 = min(c, tiles), so that c >= tiles gives every CTA exactly
 * one tile and small c many tiles per CTA (the output must not depend on it); negative: -1.
 * *pipe_grid_out (may be NULL) receives the grid of the pipelined launch, 0 when the op launched none.
 * `batch` images:
 *   op                        iargs                                         fargs   bufs
 *   FDES_B200_SWEEP_GEOM      -                                             -       int[5] out: N lo_end hi_start
 *                                                                                   line_points pipelined (no device)
 *   FDES_B200_SWEEP_DENSITY   slice slice2 nZ nslices cfg_stride cfg_off2   -       A [batch*nZ] out, rowptr (int,
 *     (S1)                    nconf rec_stride                                      [nconf][nslices*nZ*N + 1]),
 *                                                                                   col (int), w [nconf][rec_stride]
 *   FDES_B200_SWEEP_POTENTIAL slice slice2 nZ nslices cfg_stride cfg_off2   -       B [batch] out, A [batch*nZ],
 *     (S2)                    nconf                                                 Gq [nZ][(N/2+1)^2], rowptr (int)
 *   FDES_B200_SWEEP_TRANSMIT  npair                                         imPot   W [batch], D [2*batch] out
 *   FDES_B200_SWEEP_BANDLIMIT npair                                         -       W [npair ? 2*batch : batch] in/out
 *   FDES_B200_SWEEP_MULTIPLY  e_stride (images) psi_full                    -       Psi [batch] in/out, E
 *   FDES_B200_SWEEP_PROPAGATE -                                             -       Psi [batch] in/out, Pq [(N/2+1)^2]
 *   FDES_B200_SWEEP_PROPAGATE_FROM src_img_stride src_images times_n        -       out [batch], src [src_images],
 *                                                                                   Pq, lens [N*N] or 0 words (none)
 *   FDES_B200_SWEEP_COLS_FFT  ColOp dir [in_place]                          scale   in [batch], out [batch]
 *                                                                                   (float for the DP), table;
 *                                                                                   in_place (COL_PLAIN,
 *                                                                                   COL_MUL_REAL_INV): in is out
 *   FDES_B200_SWEEP_ROWS_FFT_SUM RowEpilogue band_only_in                   scale   in [batch], out (inverse)
 *   FDES_B200_SWEEP_ROWS_FFT  dir RowEpilogue in_is_real band_only_in       scale   in [batch] (float [batch][N][N]
 *                             band_only_out dn1 dn2 n1 n2 in_place                  when in_is_real), out: [batch]
 *                                                                                   (STORE, ACCUM, STORE_SHIFT),
 *                                                                                   float [batch][N][N] (INTENS_ACCUM),
 *                                                                                   float [batch][n2][n1] (CROP_REAL);
 *                                                                                   in_place (ROW_STORE, complex
 *                                                                                   input): in is out
 *   FDES_B200_SWEEP_PROBE     -                                             -       Psi [batch] out, PSI0 [1],
 *                                                                                   shifts [batch][2]
 *   FDES_B200_SWEEP_DETECTOR  ndet (1..8)                                   d1 d2   Psi [batch], out [batch][ndet]
 *                                                                           weight  (accumulated into); partial
 *                                                                           in2[ndet] sums start as NaN
 *                                                                           out2[ndet]
 *   FDES_B200_SWEEP_DETECTOR4D Q bin                                        weight  Psi [batch], out [batch][Q/bin]
 *                                                                                   [Q/bin] (accumulated into); the
 *                                                                                   [batch][Q][Q] scratch starts as
 *                                                                                   NaN in the band columns
 * The set-up, per-pixel and atom kernels, each through its production launcher (no FFT size needed; N is the
 * grid size unless noted; pi is the engine's 3.1415927f):
 *   FDES_B200_SCATTER_TABLE   Z (kirkland_row: 1..103, else the          d1 d2   Gq [(N/2+1)^2] out, [|kx|][|ky|]
 *                             unknown-element fallback)                   sigma   (ky fastest)
 *   FDES_B200_PROP_TABLE      -                                     d1 d2 d3 lambda Pq [(N/2+1)^2] out
 *   FDES_B200_LENS_TABLE      mode transposed                       ab0[14] ab1[14] tab [N*N] out ([ky][kx]; [kx][ky]
 *                                                                   defocus spread  when transposed)
 *                                                                   lambda d1 d2
 *                                                                   ObjAp extra_scale
 *   FDES_B200_DETECTOR_TABLE  mode use_incoherence use_mtf          mtfa mtfb mtfc  tab float [N*N] out
 *                                                                   mtfd illangle
 *                                                                   defocus lambda
 *                                                                   d1 d2 scale
 *   FDES_B200_TILT_BEAM       flag (+1 / -1)                        d1 d2 lambda    psi [N*N] in/out
 *                                                                   tb_x tb_y
 *   FDES_B200_TUKEY           dn1 dn2 (0..N)                        -       psi [N*N] in/out
 *   FDES_B200_AREA_MASK       dn1 dn2 (0..N)                        -       psi [N*N] in/out
 *   FDES_B200_NORM2           - (N = elements)                      -       p [N] (complex), out: the double sum of
 *                                                                           |p|^2 in 2 words
 *   FDES_B200_PEER_SUM        nsrc (1..15) (N = floats)             -       dst float [N] in/out, src_1..src_nsrc [N]
 *   FDES_B200_JITTER          (burn, nconf) pairs (N = atoms):      -       xyz [N][3], dwf [N], out [sum nconf][N][3]
 *                             streams curand_init(1, i, 0), i < 3N,         (the calls' configurations in order)
 *                             then one launch_atom_jitter per pair;
 *                             burn < 0: the streams start again
 *   FDES_B200_ANSCOMBE        seed (N = pixels)                     dose    f [N] in/out (complex, real part
 *                                                                           used), optional f2 [N]: a second call
 *                                                                           on the same streams (0 words: none)
 *   FDES_B200_RECORDS         m3 nZ nconf (N = m1 = m2)             d1 d2   xyz [nconf][nAt][3], zidx (int) [nAt],
 *                             launch_build_records as the engine    d3      occ [nAt], keys (uint), cols (int), w
 *                             runs it: binning, sort, row pointers,         [nconf][4 nAt] out, rowptr (int)
 *                             row masks (where the size has them)           [nconf][rp_stride] out, rp_stride = nkeys
 *                                                                           + 1 + mask words, nkeys = m3 nZ N
 *   FDES_B200_PLANE_WAVE      - (batch images)                      -       Psi [batch][N*N] out
 *   FDES_B200_ZERO_OUTBAND    lo_end hi_start (batch images)        -       Psi [batch][N*N] in/out
 *   FDES_B200_ABSORPTIVE      - (N = elements)                      imPot   V [N] in/out (complex)
 *   FDES_B200_SCALE_CPX       - (N = elements)                      s       p [N] in/out (complex) */
#define FDES_B200_SWEEP_GEOM 0
#define FDES_B200_SWEEP_DENSITY 1
#define FDES_B200_SWEEP_POTENTIAL 2
#define FDES_B200_SWEEP_TRANSMIT 3
#define FDES_B200_SWEEP_BANDLIMIT 4
#define FDES_B200_SWEEP_MULTIPLY 5
#define FDES_B200_SWEEP_PROPAGATE 6
#define FDES_B200_SWEEP_PROPAGATE_FROM 7
#define FDES_B200_SWEEP_COLS_FFT 8
#define FDES_B200_SWEEP_ROWS_FFT_SUM 9
#define FDES_B200_SWEEP_ROWS_FFT 10
#define FDES_B200_SWEEP_PROBE 11
#define FDES_B200_SWEEP_DETECTOR 12
#define FDES_B200_SWEEP_DETECTOR4D 13
#define FDES_B200_SCATTER_TABLE 14
#define FDES_B200_PROP_TABLE 15
#define FDES_B200_LENS_TABLE 16
#define FDES_B200_DETECTOR_TABLE 17
#define FDES_B200_TILT_BEAM 18
#define FDES_B200_TUKEY 19
#define FDES_B200_AREA_MASK 20
#define FDES_B200_NORM2 21
#define FDES_B200_PEER_SUM 22
#define FDES_B200_JITTER 23
#define FDES_B200_ANSCOMBE 24
#define FDES_B200_RECORDS 25
#define FDES_B200_PLANE_WAVE 26
#define FDES_B200_ZERO_OUTBAND 27
#define FDES_B200_ABSORPTIVE 28
#define FDES_B200_SCALE_CPX 29
int fdes_b200_sweep_test(int op, int N, int batch, const int* iargs, int n_iargs, const float* fargs, int n_fargs,
                         float** bufs, const long long* buf_elems, int nbufs, int gpu_index, int pipe_ctas,
                         int* pipe_grid_out);

#ifdef __cplusplus
}
#endif
#endif /* FDES_B200_H */
