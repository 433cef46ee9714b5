// fdes_b200 -- launch interface of the sm_100a multislice kernels (kernels.cu).
// Everything here is plain device pointers + sizes; the engine (engine.cu) owns the memory.
#pragma once
#include "launch.cuh"
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <vector>

namespace fdes {

typedef float2 cpx;

// Geometry shared by all sweeps of one simulation (square grid, N = m1 = m2).
struct SweepGeom {
    int N;              // grid size (power of two, 64..4096)
    int lo_end;         // columns kx in [0, lo_end) or [hi_start, N) can be non-zero after the
    int hi_start;       //   2/3 band limit (bounds rounded outwards to multiples of 32)
    const cpx* tw;      // pass twiddle tables of make_twiddles(N) (layout: fft_core.cuh)
    // Row masks of the deposit records (launch_row_masks): the masks of a configuration start mask_off
    // 32-bit words after its row pointers (0: none, the generic sweeps read the row pointers instead)
    int mask_off = 0;
};
// host copy of the twiddle tables a SweepGeom of size N must point to (on the device)
std::vector<cpx> make_twiddles(int N);
// the geometry every sweep of size N expects: band columns of the 2/3 limit where the register-resident
// sweeps run (the compiled bounds Band<N> of sweep_kernels.cuh check against these), every column
// (lo_end = hi_start = N) on the generic sweeps; throws for an unsupported N
SweepGeom make_sweep_geom(int N, const cpx* tw, int mask_off);

bool fft_size_supported(int N);
bool fft_size_is_fast(int N);   // register-resident kernels (else the generic run-time-N sweeps)
int rows_per_block(int N);
int cols_per_block(int N);
bool sweeps_pipelined(int N);   // column sweeps on the TMA pipeline (col_pipe.cuh): launch_propagate_cols_from works
int line_points(int N);         // points per thread E of a line transform (0: generic sweeps, no row masks)
// Grid of the pipelined column sweeps, per host thread (defined in sweeps.cu).  pipe_cta_cap 0 (the default, never
// changed by the engine): one persistent CTA per SM; c >= 1: min(c, tiles) CTAs, any number of tiles per CTA -- the
// sweep test hook sets it to run the same sweep under other tile schedules.  pipe_last_grid: the grid of the
// thread's last pipelined launch.
extern thread_local int pipe_cta_cap;
extern thread_local int pipe_last_grid;

// ---- per-slice sweeps (S1..S6, see DESIGN.md) -------------------------------------------
// The potential sweeps S1..S3 work on slice PAIRS: the densities of slice and slice2 travel as the
// real and imaginary part of one complex field (slice2 < 0: no partner).
// Image b of a launch packs slice `slice` of configuration bA = b * cfg_stride (real part) and slice `slice2`
// of configuration bB = bA + cfg_off2 (imaginary part): (1, 0) = two consecutive slices of one configuration;
// (2, 1) with slice2 == slice = the odd last slices of two configurations sharing a transform.
// S1: per-species density rows from the sorted deposit records -> row FFT -> A
void launch_density_rows(const SweepGeom& g, cpx* A, const int* rowptr, const int* rec_col,
                         const float* rec_w, int slice, int slice2, int nZ, int batch, size_t rec_stride,
                         size_t rowptr_stride, cudaStream_t st, int cfg_stride = 1, int cfg_off2 = 0);
// S2: column FFT of every species, x scattering factor, species sum, inverse column FFT -> B
void launch_potential_cols(const SweepGeom& g, cpx* B, const cpx* A, const float* Gq,
                           const int* rowptr, int slice, int slice2, int nZ, int batch, size_t rowptr_stride,
                           cudaStream_t st, int cfg_stride = 1, int cfg_off2 = 0);
// S3: inverse row FFT of W -> V_a + i V_b; per slice p < npair: exp(i V_p (1 + i imPot)) -> row FFT
//     -> D[2 b + p] (band columns only)
void launch_transmit_rows(const SweepGeom& g, const cpx* W, cpx* D, int npair, float imPot, int batch,
                          cudaStream_t st);
// S4: column FFT -> 2/3 mask and 1/N -> inverse column FFT (in place, band columns only) on the
//     entries (b, p < npair) of a [batch][2] stack, or on a plain [batch] stack when npair == 0
void launch_bandlimit_cols(const SweepGeom& g, cpx* W, int batch, int npair, cudaStream_t st);
// S5: t = IFFT_row(E), psi = IFFT_row(Psi); Psi <- FFT_row(t * psi).  E batch stride may be 0
//     (shared transmission stack).  psi_full: Psi may have out-of-band columns (first slice).
void launch_multiply_rows(const SweepGeom& g, cpx* Psi, const cpx* E, size_t e_batch_stride,
                          int batch, bool psi_full, cudaStream_t st);
// S6: column FFT -> x Fresnel propagator (quarter table, mask and 1/N folded in) -> inverse
void launch_propagate_cols(const SweepGeom& g, cpx* Psi, const cpx* Pq, int batch, cudaStream_t st);
// S6 out of place: out[b] = IFFT_col(FFT_col(c * src[b * src_img_stride]) * P [* lens]), band columns; src is an
// image stack of src_images images of N*N elements.
//   times_n (c = N): the first slice of a plane wave needs no S5 -- psi = 1, so FFT_row(t * psi) is N times the
//     band-limited FFT_row(t) that S4 left in D;
//   lens (table [kx][ky]): the CTF of the image formation (applyLensFunction, src/multisliceSimulation.cu:614-622)
//     applied in the last slice's column transform pair, out = the CTF-filtered wave.
// Only where sweeps_pipelined(N); throws for any other size (the caller runs the separate sweeps there).
void launch_propagate_cols_from(const SweepGeom& g, cpx* out, const cpx* src, int src_img_stride, int src_images,
                                const cpx* Pq, int batch, bool times_n, const cpx* lens, cudaStream_t st);

// ---- STEM probe scan ----------------------------------------------------------------------
constexpr int MAX_DETECTORS = 8;
struct DetectorRings { int n; float in2[MAX_DETECTORS], out2[MAX_DETECTORS]; };   // |k|^2 bounds [1/m^2]
// Psi[b] <- centred probe shifted by shifts[b] = (x, y) position / (N * pixel size); PSI0 is the
// column transform of the centred probe in the (kx, y) domain
void launch_probe_cols(const SweepGeom& g, cpx* Psi, const cpx* PSI0, const float* shifts, int batch,
                       cudaStream_t st);
// out[b][d] += weight * (diffraction intensity of Psi[b] inside ring d); partial: scratch of
// batch * detector_tiles(g) * MAX_DETECTORS floats
int detector_tiles(const SweepGeom& g);
void launch_detector_cols(const SweepGeom& g, const cpx* Psi, float* partial, float* out, const DetectorRings& rings,
                          float d1, float d2, float weight, int batch, cudaStream_t st);
// 4D-STEM: out[b][y][x] += weight * (sum of the bin x bin pixels (y, x) of the diffraction intensity of Psi[b],
// fftshifted and cropped to the centred window [o, o + Q)^2, o = (N - Q) / 2); out is [batch][Q/bin][Q/bin].
// scratch: [batch][Q][Q] floats, zero in the columns outside the band (the sweep writes the band columns only).
// Q = N (mod 2), bin divides Q, 1 <= Q <= N (stem4d_window, engine.h).
void launch_detector4d_cols(const SweepGeom& g, const cpx* Psi, float* scratch, float* out, int Q, int bin, float weight,
                            int batch, cudaStream_t st);
// the finish of launch_detector4d_cols: the bins of scratch summed in a fixed order (row by row) onto out
void launch_detector4d_finish(const float* scratch, float* out, int Q, int bin, float weight, int batch, cudaStream_t st);

// ---- generic sweeps used outside the slice loop ------------------------------------------
enum RowEpilogue {
    ROW_STORE = 0,         // out = scale * v
    ROW_ACCUM = 1,         // out += scale * v                      (exit-wave average)
    ROW_INTENS_ACCUM = 2,  // outI += scale * |v|^2  (float array)  (image intensity)
    ROW_STORE_SHIFT = 3,   // out[(y+N/2)%N][(x+N/2)%N] = scale * v (fftshift)
    ROW_CROP_REAL = 4      // outI[(y-dn2)*n1 + (x-dn1)] = scale * Re v inside the crop
};
struct RowOpts {
    float scale = 1.f;
    int dn1 = 0, dn2 = 0, n1 = 0, n2 = 0;   // ROW_CROP_REAL
    bool in_is_real = false;                // input is a float array (imag = 0)
    bool band_only_in = false;              // load only band columns (others are 0)
    bool band_only_out = false;             // ROW_STORE: write 0 outside the band
};
// dir = -1 forward, +1 inverse (unnormalised).  in/out batch strides are N*N elements.
void launch_rows_fft(const SweepGeom& g, const void* in, void* out, int dir, RowEpilogue epi,
                     const RowOpts& o, int batch, cudaStream_t st);

// batch-summing variant (fixed order b = 0..nb-1): out (+)= sum_b epilogue(FFT_dir(in[b])), for the
// inverse transform with ROW_ACCUM (complex out) or ROW_INTENS_ACCUM (float out)
void launch_rows_fft_sum(const SweepGeom& g, const cpx* in, void* out, int dir, RowEpilogue epi,
                         const RowOpts& o, int nb, cudaStream_t st);

enum ColOp {
    COL_PLAIN = 0,        // out = FFT_dir(in)
    COL_MUL_CPX_INV = 1,  // out = IFFT( FFT(in) * tab_c[kx][ky] )      (lens function / CTF; table stored ky-fastest;
                          // `in` must be zero outside the band columns, and only those columns of `out` are defined)
    COL_MUL_REAL_INV = 2, // out = IFFT( FFT(in) * tab_r[ky][kx] )      (MTF / incoherence)
    COL_DP_ACCUM = 3      // outI[fftshift(ky,kx)] += scale * |FFT(in)|^2   (diffraction pattern)
};
void launch_cols_fft(const SweepGeom& g, const cpx* in, void* out, int dir, ColOp op,
                     const void* table, float scale, int batch, cudaStream_t st);

// ---- set-up kernels (tables follow the reference's float32 expressions) ------------------
struct KirklandRow { float v[12]; };  // a0 b0 a1 b1 a2 b2 c0 d0 c1 d1 c2 d2
// parameters of atomic number Z (kirkland_table.inc, Z = 1..103); any other Z: the reference's unknown-element
// fallback a = 0, b = 1, c = 1, d = 0 (src/projectedPotential.cu:2984-3009)
KirklandRow kirkland_row(int Z);
// Gq[(N/2+1)^2]: scattering factor * sinc correction * normalisation (projectedPotential_d +
// divideBySinc, reference src/projectedPotential.cu:30-73, src/crystalMaker.cu:136-158)
void launch_scattering_table(float* Gq, int N, KirklandRow kr, float d1, float d2, float sigma,
                             float pi, cudaStream_t st);
// Pq[(N/2+1)^2]: Fresnel propagator with 2/3 mask and 1/N (src/multisliceSimulation.cu:253-274,
// 594-603)
void launch_propagator_table(cpx* Pq, int N, float d1, float d2, float d3, float lambda, float pi,
                             cudaStream_t st);
struct LensParams {
    float ab0[14], ab1[14];  // C1 A1 A2 B2 C3 A3 S3 A4 B4 D4 C5 A5 R5 S5
    float defocus_k, defocspread, lambda, d1, d2, ObjAp, pi;
    int mode;
};
// full [N][N] complex table of multiplyLensFunction (src/multisliceSimulation.cu:277-343);
// 0 outside the aperture; extra_scale folded in.
// transposed: entry (kx, ky) at kx * N + ky -- the layout COL_MUL_CPX_INV reads (a column's threads walk ky)
void launch_lens_table(cpx* tab, int N, const LensParams& lp, float extra_scale, cudaStream_t st, bool transposed = false);
// full [N][N] real table: MTF * (optional spatial incoherence) * scale
// (src/multisliceSimulation.cu:362-442)
struct DetectorParams {
    float mtfa, mtfb, mtfc, mtfd, illangle, defocus_k, lambda, d1, d2, pi;
    int mode; int use_incoherence;
    int use_mtf = 1;   // 0: incoherence envelope only (the stage before the noise, src/crystalMaker.cu:591-599)
};
void launch_detector_table(float* tab, int N, const DetectorParams& dp, float scale, cudaStream_t st);

// ---- small utilities ----------------------------------------------------------------------
void launch_fill_cpx(cpx* p, size_t n, cpx v, cudaStream_t st);
void launch_fill_f32(float* p, size_t n, float v, cudaStream_t st);
// plane wave psi = 1 in the (kx, y) domain (Psi = FFT_row(psi)/N): Psi[y][0] = 1, rest 0
void launch_plane_wave_rowspace(cpx* Psi, int N, int batch, cudaStream_t st);
void launch_scale_cpx(cpx* p, size_t n, float s, cudaStream_t st);
// V <- V.x * (1 + i imPot): the absorptive factor of squareAtoms_d (src/crystalMaker.cu:100-119)
// applied to a potential that was computed from the real density
void launch_absorptive_factor(cpx* V, size_t n, float imPot, cudaStream_t st);
// Psi[y][kx] = 0 for the columns outside the band (kx in [lo_end, hi_start))
void launch_zero_outband(cpx* Psi, int N, int lo_end, int hi_start, int batch, cudaStream_t st);
// deterministic sum of |p|^2 in double (two-stage tree); result[0] on device
void launch_norm2(const cpx* p, size_t n, double* partial, double* result, cudaStream_t st);
// real-space pointwise ops for the rarely used beam-tilt / Tukey / area-mask paths
void launch_tilt_beam(cpx* psi, int N, float d1, float d2, float lambda, float tb_x, float tb_y,
                      float pi, int flag, cudaStream_t st);
void launch_tukey_window(cpx* psi, int N, int dn1, int dn2, float pi, cudaStream_t st);
void launch_area_mask_blend(cpx* psi, int N, int dn1, int dn2, cudaStream_t st);

// Poisson noise through the Anscombe transform on the real part of f (ascombeNoise_d,
// src/crystalMaker.cu:50-70); states: XORWOW streams curand_init(1 + n3, pixel, 0) (:295)
void launch_anscombe_noise(cpx* f, size_t n, float dose, void* states, cudaStream_t st);

// dst[i] += sum_r src.p[r][i] (fixed order); the sources may live on peer devices that the current
// device can access (NVLink peer mappings)
constexpr int MAX_PEERS = 15;
struct PeerSources { int n; const float* p[MAX_PEERS]; };
void launch_peer_sum(float* dst, const PeerSources& src, size_t n, cudaStream_t st);

// ---- atoms: tilt, frozen phonons, binning, sort, row pointers -----------------------------
struct BinGeom {
    int m1, m2, m3, nZ;
    float d1, d2, d3;
};
void launch_rot(float* xyz, int nAt, int axA, int axB, float c, float s, cudaStream_t st);
// XORWOW states: curand_init(seed, i, 0) for i < n  (reference src/crystalMaker.cu:28-35)
size_t rng_state_bytes();
void launch_rng_init(void* states, int n, unsigned long long seed, cudaStream_t st);
// xyz_out[i] = xyz_in[i] + N(0,1) * 0.112539540f * sqrtf(dwf[i/3]); burn: draws to discard first
// for nconf consecutive configurations: xyz_out [nconf][nAt][3]
void launch_atom_jitter(float* xyz_out, const float* xyz_in, const float* dwf, int nAt,
                        void* states, long long burn, int nconf, cudaStream_t st);
// per atom: 4 deposit records (key = (i3*nZ + zidx)*m2 + row, col, weight) and the integer bin
// tuple (i1, i2, i3, zidx; -1 when rejected) -- squareAtoms_d, src/crystalMaker.cu:73-134
// nconf configurations per launch: xyz [nconf][nAt][3], records [nconf][4 nAt] (bins_out: nconf = 1)
void launch_bin_atoms(const float* xyz, const int* zidx, const float* occ, int nAt,
                      const BinGeom& bg, uint32_t* keys, int* cols, float* w, int* bins_out,
                      int nconf, cudaStream_t st);
// stable LSD radix sort of (key, col, w) by key; tmp buffers same sizes; hist: 256*nblocks ints
struct SortBuffers {
    uint32_t *keys, *keys_tmp;
    int *cols, *cols_tmp;
    float *w, *w_tmp;
    unsigned int* hist;   // 256 * sort_num_blocks(n) entries per configuration
};
int sort_num_blocks(int n);
// nconf independent arrays of n records each, stored back to back (tmp and hist likewise)
void launch_radix_sort(const SortBuffers& sb, int n, int key_bits, int nconf, cudaStream_t st);
// rowptr[k] = first sorted record with key >= k, k in [0, nkeys]; records with key >= nkeys
// (rejected atoms) stay beyond rowptr[nkeys]
// Row masks: for every configuration and every key group kg = slice * nZ + z (N consecutive keys) T = N / E
// words; bit m of word theta <-> row theta + m * T has deposit records.  These are the rows S1 writes and
// the only rows S2 may read; a thread of a column sweep holds exactly the rows of one word.
// rowptr: [nconf][rp_stride] ints, the masks of a configuration follow its nkeys + 1 row pointers.
void launch_row_masks(int* rowptr, size_t rp_stride, int nkeys, int N, int E, int nconf, cudaStream_t st);
void launch_row_pointers(const uint32_t* keys_sorted, int n, int* rowptr, int nkeys, int nconf,
                         cudaStream_t st, size_t rp_stride = 0);   // rp_stride 0: nkeys + 1
// The deposit records of nconf configurations as the slice loop reads them: binning of xyz [nconf][nAt][3] into
// sb.keys / cols / w [nconf][4 nAt], the stable sort (key_bits: bits of the largest key, nkeys = m3 * nZ * m2),
// row pointers and, when mask_E > 0, the row masks of an N = bg.m1 grid; rowptr: [nconf][rp_stride]
void launch_build_records(const float* xyz, const int* zidx, const float* occ, int nAt, const BinGeom& bg,
                          const SortBuffers& sb, int* rowptr, size_t rp_stride, int key_bits, int mask_E, int nconf,
                          cudaStream_t st);

}  // namespace fdes
