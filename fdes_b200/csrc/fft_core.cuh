// fdes_b200 -- register/shared-memory Stockham line FFT for sm_100a (complex float32).
//
// One "line" (a grid row or a grid column) of N points is transformed by T = N/E threads that
// each keep E points in registers at positions theta + m*T (m = 0..E-1).  A transform is a
// sequence of radix-R passes (R = the largest divisor of E that divides what is left; E = 20 with
// radix-5 butterflies serves the 2^a 5^b grids 320, 800, 1000 of the reference's examples).  In a
// pass a thread performs E/R radix-R DFTs on registers; between passes the line is exchanged
// through padded shared memory (Stockham autosort: natural order in, natural order out).  The
// register layout before the first pass and after the last pass is the same, so
//   * global loads/stores are coalesced (consecutive threads <-> consecutive points), and
//   * transforms can be chained (inverse -> pointwise op -> forward) with the data staying in
//     registers -- this is what lets a whole multislice sweep touch HBM once.
// With E = 32 a 1024-point line is 32 x 32: ONE shared-memory exchange per transform and, for a
// row, one warp per line (warp-level synchronisation only).
//
// Arithmetic uses the packed f32x2 instructions of sm_100 (add/mul/fma.rn.f32x2 -> FADD2 / FMUL2 /
// FFMA2): a complex add is one instruction and a complex multiply two, which halves the issue
// slots the butterflies need (the FP32 lanes themselves run at the same rate, measured with
// tools/microbench/f32x2_rate.cu).
// The index algebra is checked on the CPU by tools/fft_model.py.
//
// Replaces the cuFFT C2C calls of the reference hot path (cufftExecC2C at
// src/crystalMaker.cu:527,531 and src/multisliceSimulation.cu:554,556,608,610).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace fdes {

typedef float2 cpx;

// ---------------------------------------------------------------------------------------------
// packed f32x2 arithmetic
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ cpx padd(cpx a, cpx b)
{
    cpx c;
    asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rc, ra, rb; "
        "mov.b64 {%0,%1}, rc;}" : "=f"(c.x), "=f"(c.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return c;
}
__device__ __forceinline__ cpx psub(cpx a, cpx b)
{
    cpx c;
    asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; sub.rn.f32x2 rc, ra, rb; "
        "mov.b64 {%0,%1}, rc;}" : "=f"(c.x), "=f"(c.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return c;
}
__device__ __forceinline__ cpx pmul(cpx a, cpx b)
{
    cpx c;
    asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mul.rn.f32x2 rc, ra, rb; "
        "mov.b64 {%0,%1}, rc;}" : "=f"(c.x), "=f"(c.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return c;
}
__device__ __forceinline__ cpx pfma(cpx a, cpx b, cpx c)
{
    cpx d;
    asm("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; "
        "fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0,%1}, rd;}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}

// Loads that stay where they are written: the asm is volatile, so the compiler can neither hoist
// them above a preceding synchronisation nor batch them ahead of the transform before them
// (invariant / __restrict__ loads get hoisted to the top of the kernel and then pin 2 registers
// per element across a whole FFT).
__device__ __forceinline__ cpx ld_nc(const cpx* p)    // read-only data (tables)
{
    cpx v;
    asm volatile("ld.global.nc.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
// same with a compile-time element offset folded into the address (one base register for a
// whole unrolled sequence instead of one 64-bit pointer per load)
template <int OFF>
__device__ __forceinline__ cpx ld_nc_at(const cpx* p)
{
    cpx v;
    asm volatile("ld.global.nc.v2.f32 {%0,%1}, [%2+%3];" : "=f"(v.x), "=f"(v.y) : "l"(p), "n"(OFF * 8));
    return v;
}
// The quarter tables (propagator, scattering factors) are re-read by every tile of every image while the
// wave functions stream through L2 once per sweep: an evict_last policy keeps the tables resident.
__device__ __forceinline__ uint64_t l2_keep_policy()
{
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
template <int OFF>
__device__ __forceinline__ cpx ld_tab_at(const cpx* p)
{
    cpx v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0,%1}, [%2+%3], %4;" : "=f"(v.x), "=f"(v.y) : "l"(p), "n"(OFF * 8), "l"(l2_keep_policy()));
    return v;
}
// (the real scattering-factor tables of S2 are nZ x (N/2+1)^2 floats -- 50 MB for three species at 4096^2: kept
// resident they crowd the tiles out of L2, S2 1643 -> 1943 us; they take the default policy)
template <int OFF>
__device__ __forceinline__ float ld_tab_at(const float* p)
{
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1+%2];" : "=f"(v) : "l"(p), "n"(OFF * 4));
    return v;
}
template <int OFF>
__device__ __forceinline__ float ld_nc_at(const float* p)
{
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1+%2];" : "=f"(v) : "l"(p), "n"(OFF * 4));
    return v;
}
__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p)
{
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_nc(const float* p)
{
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ cpx ld_g(const cpx* p)     // data written by earlier kernels
{
    cpx v;
    asm volatile("ld.global.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ cpx cadd(cpx a, cpx b) { return padd(a, b); }
__device__ __forceinline__ cpx csub(cpx a, cpx b) { return psub(a, b); }
// a * (c + i s) = a * (c, c) + (-a.y, a.x) * (s, s): exactly FMUL2 + FFMA2 -- the broadcasts (R.F32), the
// pair swap and the lane signs (R.F32x2.LO_HI.NP) are operand modifiers in SASS.  (Written as
// a.x * (c, s) + a.y * (-s, c) the second multiplier needs a new register pair: MOV + FADD per multiply,
// which doubled the instruction count of every twiddle and table multiplication.)
__device__ __forceinline__ cpx cmul_cs(cpx a, float c, float s)
{
    return pfma(make_float2(-a.y, a.x), make_float2(s, s), pmul(a, make_float2(c, c)));
}
__device__ __forceinline__ cpx cmul(cpx a, cpx b) { return cmul_cs(a, b.x, b.y); }
// a * conj(b) = a * (b.x, b.x) + (a.y, -a.x) * (b.y, b.y)
__device__ __forceinline__ cpx cmul_conj(cpx a, cpx b)
{
    return pfma(make_float2(a.y, -a.x), make_float2(b.y, b.y), pmul(a, make_float2(b.x, b.x)));
}
// a * (c + i s) for COMPILE-TIME c, s: a * (c, c) + swap(a) * (-s, s).  In SASS the swap and the signs are
// operand modifiers (R.F32x2.LO_HI.NP), c is an immediate and (s, s) one uniform register pair, where the
// broadcast form of cmul_cs needs two different constant pairs in vector registers (2 extra MOVs per
// multiply -- a quarter of the instructions of a row sweep were such moves).
__device__ __forceinline__ cpx cmul_const(cpx a, float c, float s)
{
    return pfma(make_float2(a.y, a.x), make_float2(-s, s), pmul(a, make_float2(c, c)));
}
// a * conj(b)
// a + (DIR * i) * d   and   a - (DIR * i) * d      (DIR = -1: forward transform, W4 = -i)
template <int DIR>
__device__ __forceinline__ cpx add_di(cpx a, cpx d)
{
    return pfma(make_float2(d.y, d.x), DIR < 0 ? make_float2(1.f, -1.f) : make_float2(-1.f, 1.f), a);
}
template <int DIR>
__device__ __forceinline__ cpx sub_di(cpx a, cpx d)
{
    return pfma(make_float2(d.y, d.x), DIR < 0 ? make_float2(-1.f, 1.f) : make_float2(1.f, -1.f), a);
}
// a * (DIR * i)
template <int DIR>
__device__ __forceinline__ cpx mul_di(cpx a)
{
    return DIR < 0 ? make_float2(a.y, -a.x) : make_float2(-a.y, a.x);
}

// ---------------------------------------------------------------------------------------------
// in-register DFTs, natural order in / natural order out
// ---------------------------------------------------------------------------------------------
// cos / sin of 2 pi n / 32, n = 0..8
__device__ __forceinline__ constexpr float cos32(int n)
{
    constexpr float c[9] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                            0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                            0.19509032201612826785f, 0.f};
    // reduce n (mod 32) to the first octant pair
    n &= 31;
    if (n > 16) n = 32 - n;          // cos is even
    return n <= 8 ? c[n] : -c[16 - n];
}
__device__ __forceinline__ constexpr float sin32(int n) { return cos32(n - 8); }

// v *= exp(DIR * 2 pi i * n / 32) with compile-time n
template <int DIR, int n32>
__device__ __forceinline__ cpx mul_w32(cpx a)
{
    constexpr int n = ((n32 % 32) + 32) % 32;
    if constexpr (n == 0) return a;
    else if constexpr (n == 8) return mul_di<DIR>(a);
    else if constexpr (n == 16) return make_float2(-a.x, -a.y);
    else if constexpr (n == 24) return mul_di<-DIR>(a);
    else return cmul_const(a, cos32(n), DIR < 0 ? -sin32(n) : sin32(n));
}

// cos / sin of 2 pi n / 64, n = 0..16 (the W^{32 m} factors of the split 2048-point lines, split_twiddle)
__device__ __forceinline__ constexpr float cos64(int n)
{
    constexpr float c[17] = {1.00000000000000000000f, 0.99518472667219692873f, 0.98078528040323043058f, 0.95694033573220882438f, 0.92387953251128673848f, 0.88192126434835504956f, 0.83146961230254523567f, 0.77301045336273699338f, 0.70710678118654757274f, 0.63439328416364548779f, 0.55557023301960228867f, 0.47139673682599780857f, 0.38268343236508983729f, 0.29028467725446233105f, 0.19509032201612833135f, 0.09801714032956077016f, 0.00000000000000006123f};
    n &= 63;
    if (n > 32) n = 64 - n;          // cos is even
    return n <= 16 ? c[n] : -c[32 - n];
}
__device__ __forceinline__ constexpr float sin64(int n) { return cos64(n - 16); }
template <int DIR, int n64>
__device__ __forceinline__ cpx mul_w64(cpx a)
{
    constexpr int n = ((n64 % 64) + 64) % 64;
    if constexpr (n == 0) return a;
    else if constexpr (n == 16) return mul_di<DIR>(a);
    else if constexpr (n == 32) return make_float2(-a.x, -a.y);
    else if constexpr (n == 48) return mul_di<-DIR>(a);
    else return cmul_const(a, cos64(n), DIR < 0 ? -sin64(n) : sin64(n));
}

// cos / sin of 2 pi n / 20, for the radix-5 family (5, 10, 20)
__device__ __forceinline__ constexpr float cos20(int n)
{
    constexpr float c[6] = {1.f, 0.95105651629515357212f, 0.80901699437494742410f, 0.58778525229247312917f,
                            0.30901699437494742410f, 0.f};
    n = ((n % 20) + 20) % 20;
    if (n > 10) n = 20 - n;          // cos is even
    return n <= 5 ? c[n] : -c[10 - n];
}
__device__ __forceinline__ constexpr float sin20(int n) { return cos20(n - 5); }
template <int DIR, int n20>
__device__ __forceinline__ cpx mul_w20(cpx a)
{
    constexpr int n = ((n20 % 20) + 20) % 20;
    if constexpr (n == 0) return a;
    else if constexpr (n == 5) return mul_di<DIR>(a);
    else if constexpr (n == 10) return make_float2(-a.x, -a.y);
    else if constexpr (n == 15) return mul_di<-DIR>(a);
    else return cmul_const(a, cos20(n), DIR < 0 ? -sin20(n) : sin20(n));
}
// v *= exp(DIR * 2 pi i * n / R) with compile-time n; R divides 32 or 20
template <int DIR, int R, int n>
__device__ __forceinline__ cpx mul_wR(cpx a)
{
    if constexpr (32 % R == 0) return mul_w32<DIR, (32 / R) * n>(a);
    else return mul_w20<DIR, (20 / R) * n>(a);
}

template <int R, int DIR>
struct Dft;

template <int DIR>
struct Dft<2, DIR> {
    __device__ __forceinline__ static void run(cpx (&v)[2])
    {
        const cpx t = v[0];
        v[0] = cadd(t, v[1]);
        v[1] = csub(t, v[1]);
    }
};
template <int DIR>
struct Dft<4, DIR> {
    __device__ __forceinline__ static void run(cpx (&v)[4])
    {
        const cpx t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
        const cpx t2 = cadd(v[1], v[3]), d = csub(v[1], v[3]);
        v[0] = cadd(t0, t2);
        v[2] = csub(t0, t2);
        v[1] = add_di<DIR>(t1, d);
        v[3] = sub_di<DIR>(t1, d);
    }
};
template <int DIR>
struct Dft<5, DIR> {
    // X0 = x0 + t1 + t2; X1,4 = a -+ (DIR i) u; X2,3 = b -+ (DIR i) v  (forward: W = exp(-2 pi i / 5))
    __device__ __forceinline__ static void run(cpx (&v)[5])
    {
        constexpr float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;   // cos 72, cos 144
        constexpr float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;    // sin 72, sin 144
        const cpx t1 = cadd(v[1], v[4]), t2 = cadd(v[2], v[3]);
        const cpx t3 = csub(v[1], v[4]), t4 = csub(v[2], v[3]);
        const cpx x0 = v[0];
        v[0] = cadd(x0, cadd(t1, t2));
        const cpx a = pfma(t2, make_float2(c2, c2), pfma(t1, make_float2(c1, c1), x0));
        const cpx b = pfma(t2, make_float2(c1, c1), pfma(t1, make_float2(c2, c2), x0));
        const cpx u = pfma(t4, make_float2(s2, s2), pmul(t3, make_float2(s1, s1)));
        const cpx w = pfma(t4, make_float2(-s1, -s1), pmul(t3, make_float2(s2, s2)));
        // forward: X1 = a - i u, X4 = a + i u, X2 = b - i w, X3 = b + i w
        v[1] = add_di<DIR>(a, u);
        v[4] = sub_di<DIR>(a, u);
        v[2] = add_di<DIR>(b, w);
        v[3] = sub_di<DIR>(b, w);
    }
};
// R = R1 * R2, input index t = t1 + R1 t2, output index s = R2 s1 + s2:
//   X[R2 s1 + s2] = sum_t1 W_R1^{s1 t1} ( W_R^{s2 t1} sum_t2 W_R2^{s2 t2} x[t1 + R1 t2] )
template <int R, int DIR>
struct Dft {
    static constexpr int R1 = R % 4 == 0 ? 4 : (R % 5 == 0 ? 5 : 2), R2 = R / R1;
    static_assert(R == 8 || R == 16 || R == 32 || R == 10 || R == 20, "radix 2, 4, 5, 8, 10, 16, 20, 32");
    __device__ __forceinline__ static void run(cpx (&v)[R])
    {
        cpx y[R1][R2];
#pragma unroll
        for (int t1 = 0; t1 < R1; t1++) {
            cpx u[R2];
#pragma unroll
            for (int t2 = 0; t2 < R2; t2++) u[t2] = v[t1 + R1 * t2];
            Dft<R2, DIR>::run(u);
#pragma unroll
            for (int s2 = 0; s2 < R2; s2++) y[t1][s2] = u[s2];
        }
        twiddle_rows<1>(y);
        if constexpr (R1 > 2) twiddle_rows<2>(y);
        if constexpr (R1 > 3) twiddle_rows<3>(y);
        if constexpr (R1 > 4) twiddle_rows<4>(y);
#pragma unroll
        for (int s2 = 0; s2 < R2; s2++) {
            cpx z[R1];
#pragma unroll
            for (int t1 = 0; t1 < R1; t1++) z[t1] = y[t1][s2];
            Dft<R1, DIR>::run(z);
#pragma unroll
            for (int s1 = 0; s1 < R1; s1++) v[R2 * s1 + s2] = z[s1];
        }
    }
    template <int t1, int s2 = 1>
    __device__ __forceinline__ static void twiddle_rows(cpx (&y)[R1][R2])
    {
        if constexpr (s2 < R2) {
            y[t1][s2] = mul_wR<DIR, R, s2 * t1>(y[t1][s2]);
            twiddle_rows<t1, s2 + 1>(y);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// line transform
// ---------------------------------------------------------------------------------------------
// synchronisation of the threads that share a line buffer
struct SyncBlock { __device__ __forceinline__ void operator()() const { __syncthreads(); } };
struct SyncWarp { __device__ __forceinline__ void operator()() const { __syncwarp(); } };
struct SyncNamed {   // threads [id, count): bar.sync id, count  (count a multiple of 32)
    int id, count;
    __device__ __forceinline__ void operator()() const { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
};

// padded shared-memory index (one extra slot per E) -- conflict-free 64-bit scatter/gather
template <int E>
__device__ __forceinline__ int smpad(int i) { return i + (i / E); }
template <int E>
__host__ __device__ constexpr int line_smem_elems(int N) { return N + N / E; }

// Twiddle tables (built in double on the host, see make_twiddles in engine.cu), for a line of N
// points with E points per thread and passes of radix R_1 = E, R_2, ...:
//   pass p >= 2 with NS = R_1 ... R_{p-1}:  tab_p[t * NS + k] = exp(-2 pi i t k / (NS R_p)), t < R_p, k < NS
// stored back to back: offsets twiddle_offset<N, E>(p).
__host__ __device__ constexpr int pass_radix(int rem, int E)
{
    int r = 1;
    for (int d = 2; d <= E; d++)
        if (E % d == 0 && rem % d == 0) r = d;     // largest divisor of E that divides the rest
    return r;
}
template <int N, int E, int NS>
struct PassInfo {
    static constexpr int rem = N / NS;
    static constexpr int R = pass_radix(rem, E);
    static constexpr bool last = (rem == R);
    static_assert(R > 1, "line length must factor into divisors of E");
};
template <int N, int E, int NS = 1>
__host__ __device__ constexpr int twiddle_table_elems()
{
    using P = PassInfo<N, E, NS>;
    const int mine = NS > 1 ? P::R * NS : 0;
    if constexpr (P::last) return mine;
    else return mine + twiddle_table_elems<N, E, NS * P::R>();
}
template <int N, int E, int NS_TARGET, int NS = 1>
__host__ __device__ constexpr int twiddle_offset()
{
    using P = PassInfo<N, E, NS>;
    if constexpr (NS == NS_TARGET) return 0;
    else return (NS > 1 ? P::R * NS : 0) + twiddle_offset<N, E, NS_TARGET, NS * P::R>();
}

// Where the pass twiddle tables live: global memory (read-only path, L1/L2 resident) or a copy in
// shared memory (the pipelined column kernels, whose tile buffers leave little L1: LDS instead of LDG
// takes the twiddle reads out of the global load queue).  at<OFF>(i) = table[i + OFF].
struct TwGlobal {
    const cpx* p;
    template <int OFF>
    __device__ __forceinline__ cpx at(int i) const { return ld_nc_at<OFF>(p + i); }
};
struct TwShared {
    uint32_t addr;       // shared-window byte address of the table
    template <int OFF>
    __device__ __forceinline__ cpx at(int i) const
    {
        cpx v;
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2+%3];" : "=f"(v.x), "=f"(v.y) : "r"(addr + (uint32_t)i * 8u), "n"(OFF * 8));
        return v;
    }
};
// The second-pass twiddles of a 1024-point line with 32 points per thread (32 x 32) in registers.  Its only
// table is tab[t * 32 + k], t < 32, and thread theta < 32 reads entries k = theta only: 31 values, the same
// for every line the thread transforms.  w[t - 1] = tab[t * 32 + theta].
struct TwRegs {
    cpx w[31];
    __device__ __forceinline__ void load(const cpx* __restrict__ tab, int theta)
    {
#pragma unroll
        for (int t = 1; t < 32; t++) w[t - 1] = ld_nc(tab + t * 32 + theta);
    }
    template <int OFF>
    __device__ __forceinline__ cpx at(int) const     // the argument is theta
    {
        static_assert(OFF % 32 == 0 && OFF >= 32 && OFF < 1024, "TwRegs: second pass of a 32 x 32 line only");
        return w[OFF / 32 - 1];
    }
};

// v[t] *= tab[i0 + t * NS] (or its conjugate for the inverse transform), t = T0 .. R-1
template <int R, int NS, int DIR, int T0, class TW>
__device__ __forceinline__ void apply_pass_twiddles(cpx (&v)[R], TW tab, int i0)
{
    if constexpr (T0 < R) {
        const cpx w = tab.template at<T0 * NS>(i0);
        v[T0] = DIR < 0 ? cmul(v[T0], w) : cmul_conj(v[T0], w);
        apply_pass_twiddles<R, NS, DIR, T0 + 1>(v, tab, i0);
    }
}

template <int N, int E, int R, int NS, int DIR, bool LAST, class Sync, class TW>
__device__ __forceinline__ void fft_pass(cpx (&x)[E], cpx* __restrict__ sm, int theta, TW tw, Sync sync)
{
    constexpr int T = N / E, U = E / R;
#pragma unroll
    for (int u = 0; u < U; u++) {
        const int j = theta + u * T;
        const int k = j % NS;
        cpx v[R];
#pragma unroll
        for (int t = 0; t < R; t++) v[t] = x[u + t * U];
        if constexpr (NS > 1) apply_pass_twiddles<R, NS, DIR, 1>(v, tw, twiddle_offset<N, E, NS>() + k);
        Dft<R, DIR>::run(v);
        if constexpr (LAST) {
#pragma unroll
            for (int t = 0; t < R; t++) x[u + t * U] = v[t];
        } else {
            const int base = (j - k) * R + k;
#pragma unroll
            for (int t = 0; t < R; t++) sm[smpad<E>(base + t * NS)] = v[t];
        }
    }
    if constexpr (!LAST) {
        sync();
#pragma unroll
        for (int m = 0; m < E; m++) x[m] = sm[smpad<E>(theta + m * T)];
        sync();
    }
}

template <int N, int E, int NS, int DIR, class Sync, class TW>
struct LinePasses {
    __device__ __forceinline__ static void run(cpx (&x)[E], cpx* sm, int theta, TW tw, Sync sync)
    {
        using P = PassInfo<N, E, NS>;
        fft_pass<N, E, P::R, NS, DIR, P::last, Sync, TW>(x, sm, theta, tw, sync);
        if constexpr (!P::last) LinePasses<N, E, NS * P::R, DIR, Sync, TW>::run(x, sm, theta, tw, sync);
    }
};

// Transform one line held as x[m] = f[theta + m*N/E].  All threads sharing the line buffer must
// call it together.  sm: this line's line_smem_elems<E>(N) slots; tw: tables described above.
template <int N, int E, int DIR, class Sync, class TW>
__device__ __forceinline__ void fft_line_tw(cpx (&x)[E], cpx* sm, int theta, TW tw, Sync sync)
{
    static_assert(N >= E && N % E == 0, "line length must be a multiple of E");
    LinePasses<N, E, 1, DIR, Sync, TW>::run(x, sm, theta, tw, sync);
}
template <int N, int E, int DIR, class Sync>
__device__ __forceinline__ void fft_line(cpx (&x)[E], cpx* sm, int theta, const cpx* tw, Sync sync)
{
    fft_line_tw<N, E, DIR, Sync, TwGlobal>(x, sm, theta, TwGlobal{tw}, sync);
}

// ---------------------------------------------------------------------------------------------
// split lines: a line of N = 2 x 1024 points on the two warps w = 0, 1 of the line
// ---------------------------------------------------------------------------------------------
// With 32 points per thread a 2048-point line needs three Stockham passes (32 x 32 x 2) and two full
// exchanges between two warps (named barriers).  Folding the radix-2 step into the accesses that happen
// anyway leaves each warp a 1024-point transform of its own (32 x 32: one exchange, __syncwarp only):
//   first step of a transform taken from memory (decimation in frequency), j = lane + 32 m < N/2:
//       warp 0: a[j] = f[j] + f[j + N/2]            X[2k]     = FFT_{N/2}(a)[k]
//       warp 1: b[j] = (f[j] - f[j + N/2]) W^j      X[2k + 1] = FFT_{N/2}(b)[k]
//     (each warp reads both halves of the line; the result is held as x[m] = X[2 (lane + 32 m) + w])
//   last step of a transform that goes to memory (decimation in time), from x[m] = g[2 (lane + 32 m) + w]:
//       A = FFT_{N/2}(g even) in warp 0, B = FFT_{N/2}(g odd) in warp 1,
//       X[k] = A[k] + W^k B[k],  X[k + N/2] = A[k] - W^k B[k]
//     by a HALF exchange: warp 0 hands A[k], m >= 16, to warp 1 and takes W^k B[k], m < 16; every thread
//     then owns 16 values of k and emits X[k] and X[k + N/2] (16 STS + 16 LDS per thread, one barrier of
//     the two warps).
// W^j = exp(DIR 2 pi i j / N) is the t = 1 row of the line's own radix-2 pass table.
template <int N, int E>
__host__ __device__ constexpr int split_tw_offset() { return twiddle_offset<N, E, N / 2>() + N / 2; }

// W^j, j = lane + 32 m, as (compile-time W^{32 m}) x (per-thread W^lane) -- two register multiplications
// instead of a table load and one multiplication: S5 at 2048^2 232 -> 211 us (the table loads go through the
// same L1 as the row loads).  (The pipelined columns keep the table, in shared memory: no gain measured there.)
template <int N, int E, int DIR, int M>
__device__ __forceinline__ cpx split_twiddle(cpx v, cpx wlane)
{
    static_assert(N == 2048, "W^{32 m} = exp(2 pi i m / 64)");
    const cpx u = mul_w64<DIR, M>(v);
    return DIR < 0 ? cmul(u, wlane) : cmul_conj(u, wlane);
}
template <int N, int E, int DIR, int M, class Load>
__device__ __forceinline__ void split_dif_odd(cpx (&x)[E], int lane, Load load, cpx wlane)
{
    if constexpr (M < E) {
        const cpx d = psub(load(lane, M), load(lane, M + E));
        x[M] = split_twiddle<N, E, DIR, M>(d, wlane);
        split_dif_odd<N, E, DIR, M + 1>(x, lane, load, wlane);
    }
}
// load(lane, blk) = f[lane + 32 blk], blk = 0 .. 2E-1 (blk is a compile-time constant after unrolling)
template <int N, int E, int DIR, class TW, class Load>
__device__ __forceinline__ void split_dif(cpx (&x)[E], int w, int lane, TW tw, Load load)
{
    static_assert(N == 64 * E, "two warps of 32 threads with E points each");
    if (w == 0) {
#pragma unroll
        for (int m = 0; m < E; m++) x[m] = padd(load(lane, m), load(lane, m + E));
    } else {
        const cpx wlane = tw.template at<split_tw_offset<N, E>()>(lane);
        split_dif_odd<N, E, DIR, 0>(x, lane, load, wlane);
    }
}
template <int N, int E, int DIR, int M>
__device__ __forceinline__ void split_twiddle_all(cpx (&x)[E], cpx wlane)
{
    if constexpr (M < E) {
        x[M] = split_twiddle<N, E, DIR, M>(x[M], wlane);
        split_twiddle_all<N, E, DIR, M + 1>(x, wlane);
    }
}
// mine / other: 16 x 32 exchange slots of this warp / of the partner warp; pair_sync: barrier of the two
// warps; emit(lane, blk, lo, hi): X[lane + 32 blk] = lo, X[lane + 32 blk + N/2] = hi.
// The caller must make sure that `mine` is not rewritten before the partner has read it.
template <int N, int E, int DIR, class TW, class Sync, class Emit>
__device__ __forceinline__ void split_dit_combine(cpx (&x)[E], int w, int lane, TW tw, cpx* mine, const cpx* other,
                                                  Sync pair_sync, Emit emit)
{
    static_assert(N == 64 * E, "two warps of 32 threads with E points each");
    if (w == 0) {
#pragma unroll
        for (int m = 0; m < E / 2; m++) mine[m * 32 + lane] = x[m + E / 2];
    } else {
        split_twiddle_all<N, E, DIR, 0>(x, tw.template at<split_tw_offset<N, E>()>(lane));
#pragma unroll
        for (int m = 0; m < E / 2; m++) mine[m * 32 + lane] = x[m];
    }
    pair_sync();
    if (w == 0) {
#pragma unroll
        for (int m = 0; m < E / 2; m++) {
            const cpx b = other[m * 32 + lane];
            emit(lane, m, padd(x[m], b), psub(x[m], b));
        }
    } else {
#pragma unroll
        for (int m = E / 2; m < E; m++) {
            const cpx a = other[(m - E / 2) * 32 + lane];
            emit(lane, m, padd(a, x[m]), psub(a, x[m]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// column tiles
// ---------------------------------------------------------------------------------------------
// Per-thread view of a column sweep: which column line it transforms, and how the CTA's tile
// travels between global memory and the registers x[m] = f[(theta + m*T)][column].
template <int N, int E_, int CW_, bool STAGED_>
struct ColTile {
    static constexpr int E = E_, T = N / E_, CW = CW_;
    static constexpr bool STAGED = STAGED_;
    static constexpr int THREADS = CW * T;
    static constexpr int LSTRIDE = line_smem_elems<E>(N) + 16 / CW;   // bank-conflict-free line stride
    static constexpr int RPI = THREADS / CW;                          // tile rows moved per iteration
    static constexpr size_t SMEM = (size_t)CW * LSTRIDE * sizeof(cpx);
    using C = ColTile;
    int line, theta;     // column within the tile, position within the column
    int lc, lr;          // staged copies: column / first row handled by this thread
    cpx* smem;           // CTA tile buffer
    cpx* sm;             // this column's padded line buffer

    __device__ __forceinline__ explicit ColTile(cpx* smem_) : smem(smem_)
    {
        if constexpr (C::STAGED) { line = threadIdx.x / T; theta = threadIdx.x % T; }
        else { line = threadIdx.x % CW; theta = threadIdx.x / CW; }
        lc = threadIdx.x % CW;
        lr = threadIdx.x / CW;
        sm = smem + line * C::LSTRIDE;
    }
    // synchronisation among the threads that share a line buffer
    __device__ __forceinline__ void operator()() const
    {
        if constexpr (C::STAGED) __syncwarp();
        else __syncthreads();
    }
    // x[m] <- tile(theta + m*T, line); tile = &array[0][first column of the tile].
    // keep(i) == false: row mask_pos() + i*T reads as zero without touching memory (a row-mask word
    // of position mask_pos(), kernels.cuh).  `again`: the tile buffer was used by a previous
    // load/transform of this CTA.
    // position (within a line) of the rows this thread moves in load(): rows mask_pos() + i*T
    __device__ __forceinline__ int mask_pos() const { return C::STAGED ? lr : theta; }
    template <class Keep>
    __device__ __forceinline__ void load(cpx (&x)[E], const cpx* __restrict__ tile, Keep keep, bool again = false) const
    {
        if constexpr (C::STAGED) {
            if (again) __syncthreads();
            cpx v[E];
#pragma unroll
            for (int i = 0; i < E; i++) {
                const int row = lr + i * C::RPI;
                v[i] = keep(i) ? tile[(size_t)row * N + lc] : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < E; i++) smem[lc * C::LSTRIDE + smpad<E>(lr + i * C::RPI)] = v[i];
            __syncthreads();
#pragma unroll
            for (int m = 0; m < E; m++) x[m] = sm[smpad<E>(theta + m * T)];
            __syncwarp();
        } else {
#pragma unroll
            for (int m = 0; m < E; m++) {
                const int row = theta + m * T;
                x[m] = keep(m) ? tile[(size_t)row * N + line] : make_float2(0.f, 0.f);
            }
        }
    }
    __device__ __forceinline__ void store(const cpx (&x)[E], cpx* __restrict__ tile) const
    {
        if constexpr (C::STAGED) {
#pragma unroll
            for (int m = 0; m < E; m++) sm[smpad<E>(theta + m * T)] = x[m];
            __syncthreads();
            cpx v[E];
#pragma unroll
            for (int i = 0; i < E; i++) v[i] = smem[lc * C::LSTRIDE + smpad<E>(lr + i * C::RPI)];
#pragma unroll
            for (int i = 0; i < E; i++) tile[(size_t)(lr + i * C::RPI) * N + lc] = v[i];
        } else {
#pragma unroll
            for (int m = 0; m < E; m++) tile[(size_t)(theta + m * T) * N + line] = x[m];
        }
    }
};

}  // namespace fdes
