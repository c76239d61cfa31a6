// gsc_kernels.cuh -- every kernel of the frame pipeline except the online
// k-means (gsc_online.cuh).  One translation unit (gsc_api.cu) includes all.
//
// Stage map (SURVEY.md section 2, "New kernel" table):
//   K2 k_find_divider        enc:566-605
//   K1 k_make_chunks         enc:326-439, 349-363, 258-322, 1700-1716
//   K3 k_seed_*              yakmo init() / run(0)  (enc:824-828)
//   K5 k_owner_sums          cell sums / class means in point order (enc:845-864)
//   K7 k_dictionary          enc:865-882 (+ passthrough enc:891-912)
//   K6 k_knnfit              enc:928-965
//      k_finalize            enc:970-977
//   Lloyd: k_assign (+ k_owner_sums) ; legacy ANN: k_ann_*
#pragma once
#include "gsc_device.cuh"
#include "gsc_log.h"

// ---------------------------------------------------------------------------
// Constant tables: trig tables are computed on the HOST with libm so that
// they are the very doubles the reference's cos()/sin() calls produce on this
// machine (enc:270-271, 292-293, 1712); uploaded once per chunk size.
// ---------------------------------------------------------------------------
struct GscTrig {
    double dct[GSC_MAX_CS * GSC_MAX_CS];  // cos(pi/cs*(n+0.5)*k)      [k][n]
    double dc[GSC_MAX_CS * GSC_MAX_CS];   // cos(-2*pi*k*i/cs)         [k][i]
    double ds[GSC_MAX_CS * GSC_MAX_CS];   // sin(-2*pi*k*i/cs)
    double ic[GSC_MAX_CS * GSC_MAX_CS];   // cos( 2*pi*k*i/cs)
    double is[GSC_MAX_CS * GSC_MAX_CS];   // sin( 2*pi*k*i/cs)
    double s0;                            // sqrt(0.5)
    double scale;                         // sqrt(2.0/cs)
};
__constant__ GscTrig c_trig_all[3];  // chunk size 2, 4, 8
template <int CS> struct GscTrigIdx { static constexpr int v = (CS == 2) ? 0 : (CS == 4) ? 1 : 2; };
#define c_trig (c_trig_all[GscTrigIdx<CS>::v])

// ---------------------------------------------------------------------------
// K2  FindAttenuationDivider (enc:566-605)
// One CTA of 64 threads per frame: thread t evaluates divider t+1 over the
// whole frame in the reference's order (channel -> chunk -> sample), so the
// Double sum v is the reference's sum bit for bit.  Thread-level parallelism
// comes from the 64 dividers x the frames of the batch.
// ---------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(64) k_find_divider(const GscFrame *__restrict__ frames,
                                                     const short *__restrict__ pcm, int bits,
                                                     int *__restrict__ divider_out,
                                                     double *__restrict__ v_out) {
    const GscFrame f = frames[blockIdx.x];
    const int t = threadIdx.x;
    const double law = 1.0 / (double)(t + 1);
    GscLaw L;
    L.init(law);
    const int obd = (1 << (bits - 1)) - 1;
    double v = 0.0;
    const int nchunks = f.S / CS;
    for (int j = 0; j < f.C; ++j) {
        const short *row = pcm + f.pcm_off + (long long)j * f.stride;
        for (int k = 0; k < nchunks; ++k) {
            double x[CS];
            int hi = 0;
#pragma unroll
            for (int l = 0; l < CS; ++l) {
                x[l] = gsc_sample(row[k * CS + l]);
                int h = gsc_hi(x[l]);
                hi = h > hi ? h : hi;
            }
            const int a = gsc_attenuation(hi, L);
            const double coeff = L.T[a];
#pragma unroll
            for (int l = 0; l < CS; ++l) {
                short os = gsc_quant(x[l], obd, coeff, false);
                double fs = gsc_dequant(os, obd, coeff, false);
                double d = x[l] - fs;
                v += d * d;
            }
        }
    }
    __shared__ double sv[64];
    sv[t] = v;
    if (v_out) v_out[(long long)f.slot * 64 + t] = v;
    __syncthreads();
    if (t == 0) {
        int bestDiv = 1;
        double best = 3.40282346638528860e+38;  // MaxSingle, enc:575
        for (int i = 0; i < 64; ++i)
            if (sv[i] < best) { best = sv[i]; bestDiv = i + 1; }
        divider_out[f.slot] = bestDiv;
    }
}

// ---------------------------------------------------------------------------
// K2, second form.  Same contract (thread t = divider t+1, its Double sum formed in the reference's order), with the
// work that does not depend on the divider done once per CTA and the divisions taken out of the inner loop:
//   * a tile of 64 chunks is converted to Double (x = s / 32767.0, enc:1645) and its chunk peaks hi (enc:1687-1690)
//     computed cooperatively, then every divider thread reads them as shared-memory broadcasts;
//   * ComputeAttenuation's loop "first r with hi * T[r] > 32767" (enc:1692-1697) is monotone in hi, so each divider
//     tabulates hmax[r] = the largest integer hi that does NOT trip r (found with the very same Double predicate) and
//     the per-chunk attenuation is a 4-step search over integers;
//   * makeFloatSample's division q / (obd * coeff) (enc:1676) has only 16 distinct divisors per divider: with
//     R = RN(1 / y) tabulated, q0 = RN(q R), r = fma(-q0, y, q) (exact), q1 = fma(r, R, q0) is the correctly rounded
//     quotient (Markstein); k_check_divider_division verifies it against the hardware division for EVERY
//     (divider, attenuation, q) that can occur at 8 and 12 bits (the test runs it), other bit depths divide.
// ---------------------------------------------------------------------------
#define GSC_DIV_TILE 64
__device__ __forceinline__ double gsc_div_markstein(double q, double y, double R) {
    const double q0 = q * R;
    const double r = fma(-q0, y, q);
    return fma(r, R, q0);
}

template <int CS>
__global__ void __launch_bounds__(64) k_find_divider2(const GscFrame *__restrict__ frames, const short *__restrict__ pcm,
                                                      int bits, int *__restrict__ divider_out, double *__restrict__ v_out) {
    __shared__ double s_x[GSC_DIV_TILE * CS];
    __shared__ int s_hi[GSC_DIV_TILE];
    __shared__ double s_T[GSC_MAX_ATT + 2][64];   // coeff table of every divider, [r][divider]: conflict-free
    __shared__ double s_Y[GSC_MAX_ATT + 1][64];   // obd * coeff
    __shared__ double s_R[GSC_MAX_ATT + 1][64];   // RN(1 / (obd * coeff))
    __shared__ int s_hmax[GSC_MAX_ATT + 2][64];
    __shared__ double sv[64];
    const GscFrame f = frames[blockIdx.x];
    const int t = threadIdx.x;
    const double law = 1.0 / (double)(t + 1);
    const int obd = (1 << (bits - 1)) - 1;
    const bool fastdiv = (bits == 8 || bits == 12);
    {
        double c = 1.0 + 0.0 * law;
        s_T[0][t] = c;
        for (int r = 1; r <= GSC_MAX_ATT + 1; ++r) { c = c + (double)r * law; s_T[r][t] = c; }
        for (int a = 0; a <= GSC_MAX_ATT; ++a) { const double y = (double)obd * s_T[a][t]; s_Y[a][t] = y; s_R[a][t] = 1.0 / y; }
        for (int r = 1; r <= GSC_MAX_ATT + 1; ++r) {       // largest hi in [0, 32768] with !(hi * T[r] > 32767)
            const double T = s_T[r][t];
            int lo = 0, hi = 32769;                        // predicate false at lo (0 * T = 0), true at 32769 (T >= 1)
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if ((double)mid * T > 32767.0) hi = mid; else lo = mid; }
            s_hmax[r][t] = lo;
        }
    }
    double v = 0.0;
    const int nchunks = f.S / CS;
    for (int j = 0; j < f.C; ++j) {
        const short *row = pcm + f.pcm_off + (long long)j * f.stride;
        for (int k0 = 0; k0 < nchunks; k0 += GSC_DIV_TILE) {
            const int tc = min(GSC_DIV_TILE, nchunks - k0);
            __syncthreads();
            for (int e = t; e < tc * CS; e += 64) s_x[e] = gsc_sample(row[(long long)k0 * CS + e]);
            __syncthreads();
            if (t < tc) {
                int hi = 0;
#pragma unroll
                for (int l = 0; l < CS; ++l) { const int h = gsc_hi(s_x[t * CS + l]); hi = h > hi ? h : hi; }
                s_hi[t] = hi;
            }
            __syncthreads();
            for (int k = 0; k < tc; ++k) {
                const int hi = s_hi[k];
                // attenuation: first r in 1..15 with hi > hmax[r] (else 16), minus one  (enc:1692-1697)
                int lo_r = 1, hi_r = GSC_MAX_ATT + 1;
                while (lo_r < hi_r) { const int mid = (lo_r + hi_r) >> 1; if (hi > s_hmax[mid][t]) hi_r = mid; else lo_r = mid + 1; }
                const int a = lo_r - 1;
                const double coeff = s_T[a][t], y = s_Y[a][t], R = s_R[a][t];
#pragma unroll
                for (int l = 0; l < CS; ++l) {
                    const double x = s_x[k * CS + l];
                    const short os = gsc_quant(x, obd, coeff, false);
                    double fs = fastdiv ? gsc_div_markstein((double)os, y, R) : (double)os / y;
                    if (fs < -1.0) fs = -1.0;
                    if (fs > 1.0) fs = 1.0;
                    const double d = x - fs;
                    v += d * d;
                }
            }
        }
    }
    sv[t] = v;
    if (v_out) v_out[(long long)f.slot * 64 + t] = v;
    __syncthreads();
    if (t == 0) {
        int bestDiv = 1;
        double best = 3.40282346638528860e+38;  // MaxSingle, enc:575
        for (int i = 0; i < 64; ++i)
            if (sv[i] < best) { best = sv[i]; bestDiv = i + 1; }
        divider_out[f.slot] = bestDiv;
    }
}

// Exhaustive check of gsc_div_markstein against the division it replaces: every divider 1..64, attenuation 0..15 and
// quantised sample -obd..obd at the given bit depth.  out[0] += mismatches (bit patterns compared).
__global__ void k_check_divider_division(int bits, unsigned long long *__restrict__ out) {
    const int t = blockIdx.x;                  // divider t+1
    const double law = 1.0 / (double)(t + 1);
    const int obd = (1 << (bits - 1)) - 1;
    double T[GSC_MAX_ATT + 1];
    double c = 1.0 + 0.0 * law;
    T[0] = c;
    for (int r = 1; r <= GSC_MAX_ATT; ++r) { c = c + (double)r * law; T[r] = c; }
    unsigned long long bad = 0;
    for (int a = 0; a <= GSC_MAX_ATT; ++a) {
        const double y = (double)obd * T[a], R = 1.0 / y;
        for (int q = -obd + (int)threadIdx.x; q <= obd; q += blockDim.x) {
            const double want = (double)q / y, got = gsc_div_markstein((double)q, y, R);
            bad += (__double_as_longlong(want) != __double_as_longlong(got));
        }
    }
    if (bad) atomicAdd(out, bad);
}

// ---------------------------------------------------------------------------
// K1  chunk extraction, heuristic attributes, features (enc:467-485)
// One thread per chunk.  grid = (ceil(maxN/256), F).
// ---------------------------------------------------------------------------
template <int CS>
__device__ __forceinline__ void gsc_features(const double (&x)[CS], bool neg, bool rev,
                                             float *__restrict__ out) {
    double data[CS], temp[CS];
#pragma unroll
    for (int i = 0; i < CS; ++i) data[i] = (rev ? x[CS - 1 - i] : x[i]) * (neg ? -1.0 : 1.0);  // enc:356
#pragma unroll
    for (int k = 0; k < CS; ++k) {  // enc:1706-1715
        const double s = (k == 0) ? c_trig.s0 : 1.0;
        double sum = 0;
#pragma unroll
        for (int n = 0; n < CS; ++n) sum += s * data[n] * c_trig.dct[k * CS + n];
        out[k] = (float)(sum * c_trig.scale);
    }
#pragma unroll
    for (int k = 0; k < CS; ++k) {  // enc:258-278 DFT power
        double re = 0, im = 0;
#pragma unroll
        for (int i = 0; i < CS; ++i) {
            re += data[i] * c_trig.dc[k * CS + i];
            im += data[i] * c_trig.ds[k * CS + i];
        }
        temp[k] = re * re + im * im;
    }
#pragma unroll
    for (int i = 0; i < CS; ++i)  // enc:316-318, math.log10 = ln(x)*const; ln = the shared correctly-rounded routine
        if (!(fabs(temp[i]) <= 1e-12)) temp[i] = gsc_log_cr(temp[i]) * 0.43429448190325182765;
#pragma unroll
    for (int k = 0; k < CS; ++k) {  // enc:280-302 iDFT magnitude
        double re = 0, im = 0;
#pragma unroll
        for (int i = 0; i < CS; ++i) {
            re += temp[i] * c_trig.ic[k * CS + i];
            im += temp[i] * c_trig.is[k * CS + i];
        }
        re /= (double)CS;
        im /= (double)CS;
        out[CS + k] = (float)(sqrt(re * re + im * im) * 0.00001);  // enc:362
    }
}

template <int CS>
__global__ void __launch_bounds__(256) k_make_chunks(const GscFrame *__restrict__ frames,
                                                     const short *__restrict__ pcm, int bits,
                                                     const int *__restrict__ divider,
                                                     unsigned char *__restrict__ attr,
                                                     unsigned char *__restrict__ atten,
                                                     float *__restrict__ feat,
                                                     short *__restrict__ dst) {
    const GscFrame f = frames[blockIdx.y];
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= f.N) return;
    const int i = n / f.C, ch = n - i * f.C;
    GscLaw L;
    L.init(1.0 / (double)divider[f.slot]);  // enc:561-564
    const short *row = pcm + f.pcm_off + (long long)ch * f.stride;
    double x[CS];
#pragma unroll
    for (int l = 0; l < CS; ++l) {
        int p = i * CS + l;
        x[l] = (p < f.S) ? gsc_sample(row[p]) : 0.0;
    }
    int a; bool ng, rv;
    gsc_chunk_attrs<CS>(x, L, a, ng, rv);
    const long long g = f.chunk_off + n;
    if (attr) attr[g] = (unsigned char)((ng ? 2 : 0) | (rv ? 1 : 0));
    if (atten) atten[g] = (unsigned char)a;
    if (dst) {
        const int obd = (1 << (bits - 1)) - 1;
#pragma unroll
        for (int l = 0; l < CS; ++l) dst[g * CS + l] = gsc_quant(x[l], obd, L.T[a], ng);
    }
    if (feat) {
        float o[2 * CS];
        gsc_features<CS>(x, ng, rv, o);
        float4 *fo = reinterpret_cast<float4 *>(feat + g * 2 * CS);
        if (CS % 2 == 0) {
#pragma unroll
            for (int l = 0; l < 2 * CS / 4; ++l) fo[l] = make_float4(o[4 * l], o[4 * l + 1], o[4 * l + 2], o[4 * l + 3]);
        } else {
#pragma unroll
            for (int l = 0; l < 2 * CS; ++l) feat[g * 2 * CS + l] = o[l];
        }
    }
}

// ---------------------------------------------------------------------------
// K3  yakmo seeding (k-means++ / random), one CTA per frame.
// Faithful to init() (RVA 0x16f0): xor128-64 RNG, float norm-expansion
// distances, running FLOAT prefix sum r[] in point order, std::lower_bound,
// linear probe.  The prefix sum is the reference's sequential float chain: it
// is evaluated by warp 0 in point order (exact), everything else is parallel.
// ---------------------------------------------------------------------------
struct GscXor128 { unsigned long long x, y, z, w; };
__device__ __forceinline__ float gsc_xor128(GscXor128 &g) {
    unsigned long long t = g.x ^ (g.x << 11);
    g.x = g.y; g.y = g.z; g.z = g.w;
    g.w = (g.w ^ (g.w >> 19)) ^ (t ^ (t >> 8));
    return (float)((double)g.w * 5.42101086242752217e-20);  // 2^-64
}

template <int D>
__device__ __forceinline__ void gsc_load_row(const float *__restrict__ X, long long j, float (&p)[D]) {
    if (D % 4 == 0) {
        const float4 *v = reinterpret_cast<const float4 *>(X + j * D);
#pragma unroll
        for (int k = 0; k < D / 4; ++k) {
            float4 t = v[k];
            p[4 * k] = t.x; p[4 * k + 1] = t.y; p[4 * k + 2] = t.z; p[4 * k + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) p[k] = X[j * D + k];
    }
}

#define GSC_SEED_THREADS 512
#define GSC_SCAN_E 4                                   // elements per thread per window
#define GSC_SCAN_WIN (GSC_SEED_THREADS * GSC_SCAN_E)   // elements per window

// ---------------------------------------------------------------------------
// Exact PARALLEL evaluation of the sequential float recurrence
//     r[j] = fl(r[j-1] + a[j]),   r[-1] = +0          (yakmo: obj += up; r[j] = obj)
// Float addition is not associative, so a tree reduction gives other bits.
// But while the running sum stays inside one binade [2^E, 2^(E+1)) every
// partial sum is an integer multiple S*u of u = ulp = 2^(E-23), and
//     S_j = S_{j-1} + floor(a_j/u) + round_bit,
// where round_bit depends only on the fraction of a_j/u and, for an exact tie,
// on the PARITY of S (round half to even).  Each element is therefore a
// function  parity -> increment, those functions compose associatively, and a
// block-wide scan of them reproduces the sequential result bit for bit.
// The array is taken in aligned windows of 512 x 8 elements held in registers
// (two 128-bit loads per thread).  Inside a window the scan is repeated in
// ROUNDS: a round certifies everything up to the first element that would leave
// the binade (or is non-finite / huge); that element is added with one real
// float addition and the next round continues behind it in the new binade
// without touching memory again.  A zero running sum is skipped in parallel;
// stretches with little progress (the first few hundred elements, where the sum
// doubles every few elements) fall back to a one-warp serial chain.
// All threads of the CTA must call this; returns the final sum to everyone.
// ---------------------------------------------------------------------------
struct GscScanSmem {
    int w0[GSC_SEED_THREADS / 32], w1[GSC_SEED_THREADS / 32];
    int wv[GSC_SEED_THREADS / 32];
    unsigned long long n_rounds, n_serial;   // debug counters
    float run;      // running sum handed back by the serial chain
    float before;   // value of the sum just before the first uncertified element of the round
    float addend;   // ... and that element itself (from its owner's registers)
};

__device__ __forceinline__ void gsc_scan_compose(int &f0, int &f1, int g0, int g1) {
    // (f then g)(p) = f(p) + g((p + f(p)) & 1)
    const int h0 = f0 + ((f0 & 1) ? g1 : g0);
    const int h1 = f1 + (((1 + f1) & 1) ? g1 : g0);
    f0 = h0; f1 = h1;
}

__device__ float gsc_seq_prefix(const float *__restrict__ a, float *__restrict__ r, int N, GscScanSmem &sm) {
    constexpr int E = GSC_SCAN_E;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // running sum before element `pos`, first element not yet final, element that the last round added with a
    // real float addition (-1: none): every thread keeps its own (identical) copy
    float run = 0.0f;
    int pos = 0, addidx = -1;
    __syncthreads();
    // this thread's elements of a window (the window after the current one is fetched while the current one is
    // scanned: with hundreds of frames in flight the array comes from HBM, not from L2)
    auto load_win = [&](int wb, float (&dst)[E]) {
        const int jj = wb + tid * E;
        if ((jj + E <= N) && ((reinterpret_cast<unsigned long long>(a + jj) & 15ull) == 0ull)) {
#pragma unroll
            for (int q = 0; q < E / 4; ++q) {
                const float4 t = *reinterpret_cast<const float4 *>(a + jj + 4 * q);
                dst[4 * q] = t.x; dst[4 * q + 1] = t.y; dst[4 * q + 2] = t.z; dst[4 * q + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) dst[e] = (jj + e < N) ? a[jj + e] : 0.0f;
        }
    };
    float vnext[E];
    load_win(0, vnext);
    for (int wbase = 0; wbase < N; wbase += GSC_SCAN_WIN) {
        const int wend = min(N, wbase + GSC_SCAN_WIN);
        const int j0 = wbase + tid * E;
        const bool vec = (j0 + E <= N) && ((reinterpret_cast<unsigned long long>(r + j0) & 15ull) == 0ull);
        // this thread's elements of the window, in registers for every round
        float v[E], out[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = vnext[e];
        if (wbase + GSC_SCAN_WIN < N) load_win(wbase + GSC_SCAN_WIN, vnext);
#pragma unroll
        for (int e = 0; e < E; ++e) out[e] = 0.0f;
        for (;;) {   // rounds
            // the element the previous round added for real belongs to someone: its value is the running sum
#pragma unroll
            for (int e = 0; e < E; ++e) if (j0 + e == addidx) out[e] = run;
            if (pos >= wend) break;
            const unsigned rb = __float_as_uint(run);
            const int E0 = (int)((rb >> 23) & 0xffu);
            int viol = wend;  // first index >= pos this thread cannot certify

            if (run == 0.0f) {
                // 0 + a = a exactly: the zero run is skipped in parallel (outputs stay 0)
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int j = j0 + e;
                    if (j >= pos && j < wend && viol == wend) { if (v[e] != 0.0f) viol = j; else out[e] = 0.0f; }
                }
                __syncthreads();   // keeps the barrier count of both branches equal
            } else if ((rb >> 31) == 0u && E0 >= 24 && E0 <= 250) {
                // positive normal running sum: integer-domain scan within the binade.  a_j / ulp is formed
                // exactly in float (power-of-two scaling), split into floor and fraction; inc = round bit that
                // does not depend on parity, tie = exact half (round to even: depends on the parity of S).
                const int Sm = (int)((rb & 0x7fffffu) | 0x800000u);
                const float sc = __uint_as_float((unsigned)(277 - E0) << 23);     // 1 / ulp = 2^(150 - E0)
                const float huge = __uint_as_float((unsigned)(E0 + 2) << 23);     // 4 * 2^(E0-127): two binades up
                int I[E], cls[E];   // cls: bit0 = inc, bit1 = tie, 4 = cannot be certified
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int j = j0 + e;
                    I[e] = 0; cls[e] = 0;
                    if (j >= pos && j < wend) {
                        const float av = fabsf(v[e]);
                        if (!(av < huge)) { I[e] = 1 << 26; cls[e] = 4; }   // non-finite / huge
                        else {
                            const float aq = av * sc;         // exact, < 2^25
                            const float fl = floorf(aq);
                            const float g = aq - fl;          // exact fraction
                            const int ni = (int)fl;
                            const int tie = (g == 0.5f) ? 2 : 0;
                            if (v[e] >= 0.0f) { I[e] = ni; cls[e] = tie | ((g > 0.5f) ? 1 : 0); }
                            else if (g == 0.0f) { I[e] = -ni; }
                            else { I[e] = -(ni + 1); cls[e] = tie | ((g < 0.5f) ? 1 : 0); }   // floor(-x) = -(n+1), fraction 1 - g
                        }
                    }
                }
                // this thread's elements as a function parity -> increment (elements before pos are the identity)
                int f0 = 0, f1 = 1;   // running S (mod offset) for start parity 0 / 1
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int t0 = f0 + I[e], t1 = f1 + I[e];
                    f0 = t0 + ((cls[e] & 1) | ((cls[e] >> 1) & t0 & 1));
                    f1 = t1 + ((cls[e] & 1) | ((cls[e] >> 1) & t1 & 1));
                }
                f1 -= 1;
                // inclusive warp scan
                int s0 = f0, s1 = f1;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int p0 = __shfl_up_sync(0xffffffffu, s0, o), p1 = __shfl_up_sync(0xffffffffu, s1, o);
                    if (lane >= o) { int q0 = p0, q1 = p1; gsc_scan_compose(q0, q1, s0, s1); s0 = q0; s1 = q1; }
                }
                if (lane == 31) { sm.w0[warp] = s0; sm.w1[warp] = s1; }
                __syncthreads();
                int x0 = 0, x1 = 0;
                {
                    // composition of the warps before this one: a log-step scan of the per-warp functions over the
                    // lanes (lane w holds warp w's function) instead of a serial walk through shared memory
                    constexpr int NW = GSC_SEED_THREADS / 32;
                    int a0 = (lane < NW) ? sm.w0[lane] : 0, a1 = (lane < NW) ? sm.w1[lane] : 0;
#pragma unroll
                    for (int o = 1; o < NW; o <<= 1) {
                        const int p0 = __shfl_up_sync(0xffffffffu, a0, o), p1 = __shfl_up_sync(0xffffffffu, a1, o);
                        if (lane >= o) { int q0 = p0, q1 = p1; gsc_scan_compose(q0, q1, a0, a1); a0 = q0; a1 = q1; }
                    }
                    const int src = warp > 0 ? warp - 1 : 0;
                    const int b0 = __shfl_sync(0xffffffffu, a0, src), b1 = __shfl_sync(0xffffffffu, a1, src);
                    if (warp > 0) { x0 = b0; x1 = b1; }
                }
                {
                    int e0 = __shfl_up_sync(0xffffffffu, s0, 1), e1 = __shfl_up_sync(0xffffffffu, s1, 1);
                    if (lane == 0) { e0 = 0; e1 = 0; }
                    gsc_scan_compose(x0, x1, e0, e1);
                }
                int S = Sm + ((Sm & 1) ? x1 : x0);
                // replay own elements with the true S, certify and record
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int j = j0 + e;
                    if (j >= pos && j < wend && viol == wend) {
                        const int t = S + I[e];
                        const int Sn = t + ((cls[e] & 1) | ((cls[e] >> 1) & t & 1));
                        if (cls[e] >= 4 || t < (1 << 23) || Sn >= (1 << 24) || S < (1 << 23) || S >= (1 << 24)) viol = j;
                        else { S = Sn; out[e] = __uint_as_float(((unsigned)E0 << 23) | ((unsigned)Sn & 0x7fffffu)); }
                    }
                }
            } else {
                viol = pos;  // negative / denormal / non-finite running sum: one real addition
                __syncthreads();
            }
            // first uncertified index of the window
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) viol = min(viol, __shfl_xor_sync(0xffffffffu, viol, o));
            if (lane == 0) sm.wv[warp] = viol;
            __syncthreads();
            int vv = wend;
#pragma unroll
            for (int w = 0; w < GSC_SEED_THREADS / 32; ++w) vv = min(vv, sm.wv[w]);
            // elements [pos, vv) are final.  The owner of element vv-1 publishes the sum reached there.
            if (vv > pos) {
#pragma unroll
                for (int e = 0; e < E; ++e) if (j0 + e == vv - 1) sm.before = out[e];
            } else if (tid == 0) {
                sm.before = run;
            }
#pragma unroll
            for (int e = 0; e < E; ++e) if (j0 + e == vv) sm.addend = v[e];
            const bool serial = (run != 0.0f) && (vv - pos < 64) && (vv < wend);
            if (tid == 0) { sm.n_rounds++; if (serial) sm.n_serial++; }
            __syncthreads();
            if (serial) {
                // little progress: one-warp serial chain over the next (up to) 256 elements, from memory
                const int lim = min(wend, vv + 256);
                if (warp == 0) {
                    float rr = sm.before;
                    for (int b0 = vv; b0 < lim; b0 += 32) {
                        const int j = b0 + lane;
                        const float val = (j < lim) ? a[j] : 0.0f;
                        float mine = 0.0f;
                        const int cntl = min(32, lim - b0);
                        for (int l = 0; l < cntl; ++l) {
                            const float x = __shfl_sync(0xffffffffu, val, l);
                            rr = rr + x;
                            if (lane == l) mine = rr;
                        }
                        if (j < lim) r[j] = mine;
                    }
                    if (lane == 0) sm.run = rr;
                }
                __syncthreads();
                run = sm.run; pos = lim; addidx = -1;
                // the chain wrote r[vv .. lim): their owners take the values over (the window is stored at its end)
#pragma unroll
                for (int e = 0; e < E; ++e) { const int j = j0 + e; if (j >= vv && j < lim) out[e] = r[j]; }
            } else if (vv < wend) {
                run = sm.before + sm.addend;   // the one real float addition
                pos = vv + 1; addidx = vv;
            } else {
                run = sm.before; pos = wend; addidx = -1;
            }
        }
        // store the window
        if (vec) {
#pragma unroll
            for (int q = 0; q < E / 4; ++q)
                *reinterpret_cast<float4 *>(r + j0 + 4 * q) = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) { const int j = j0 + e; if (j < wend) r[j] = out[e]; }
        }
        __syncthreads();
    }
    __syncthreads();
    return run;
}

template <int D>
__global__ void __launch_bounds__(GSC_SEED_THREADS) k_seed(const GscFrame *__restrict__ frames,
                                                           const float *__restrict__ X,   // [sumN][D]
                                                           int init_type,
                                                           float *__restrict__ pnorm,     // [sumN]
                                                           float *__restrict__ up,        // [sumN]
                                                           float *__restrict__ r,         // [sumN]
                                                           int *__restrict__ sid,         // [sumN] seed cell
                                                           int *__restrict__ seeds,       // [F][Kmax] or null
                                                           float *__restrict__ cen,       // [F][Kmax][D] seeds out
                                                           float *__restrict__ cnorm,     // [F][Kmax]
                                                           int Kmax, int serial_scan,
                                                           unsigned long long *__restrict__ sdbg) {
    extern __shared__ unsigned chosen[];  // N bits
    __shared__ float s_c[D];
    __shared__ float s_cn;
    __shared__ float s_obj;
    __shared__ GscScanSmem s_scan;
    const GscFrame f = frames[blockIdx.x];
    const int K = f.K, N = f.N;
    if (K <= 0) return;
    const int tid = threadIdx.x;
    const float *Xf = X + f.chunk_off * D;
    float *pn = pnorm + f.chunk_off, *upf = up + f.chunk_off, *rf = r + f.chunk_off;
    int *sidf = sid + f.chunk_off;
    float *cenf = cen + (long long)f.slot * Kmax * D;
    float *cnf = cnorm + (long long)f.slot * Kmax;

    for (int w = tid; w < (N + 31) / 32; w += blockDim.x) chosen[w] = 0u;
    // load(): norm = sum v*v, left to right in float
    for (int j = tid; j < N; j += blockDim.x) {
        float p[D];
        gsc_load_row<D>(Xf, j, p);
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < D; ++k) { float m = p[k] * p[k]; s = s + m; }
        pn[j] = s;
    }
    GscXor128 g = {123456789ull, 362436069ull, 521288629ull, 88675123ull};
    if (tid == 0) { s_obj = 0.0f; s_scan.n_rounds = 0; s_scan.n_serial = 0; }
    __syncthreads();

    unsigned long long c_pick = 0, c_dist = 0, c_scan = 0, c_t = 0;
    for (int i = 0; i < K; ++i) {
        if (tid == 0) c_t = clock64();
        if (tid == 0) {
            float u = gsc_xor128(g);
            unsigned c;
            if (init_type == 0 || i == 0) {
                c = (unsigned)(long long)floorf(u * (float)N);
            } else {
                float target = u * s_obj;
                long long first = 0, count = N;
                while (count > 0) {  // std::lower_bound
                    long long half = count >> 1;
                    if (target > rf[first + half]) { first = first + half + 1; count = count - half - 1; }
                    else count = half;
                }
                c = (unsigned)first;
            }
            while (c < (unsigned)N && ((chosen[c >> 5] >> (c & 31)) & 1u))
                c = (c >= (unsigned)(N - 1)) ? 0u : c + 1u;
            if (c >= (unsigned)N) c = (unsigned)(N - 1);
            chosen[c >> 5] |= 1u << (c & 31);
            if (seeds) seeds[(long long)f.slot * Kmax + i] = (int)c;
#pragma unroll
            for (int k = 0; k < D; ++k) { float v = Xf[(long long)c * D + k]; s_c[k] = v; cenf[(long long)i * D + k] = v; }
            s_cn = pn[c];
            cnf[i] = pn[c];
        }
        __syncthreads();
        if (tid == 0) { const unsigned long long t1 = clock64(); c_pick += t1 - c_t; c_t = t1; }
        const float cn = s_cn;
        // the seed row stays in shared memory and is re-read where a row is actually scored (~5 % of the points):
        // the registers it would occupy pay for the prefetch of the next quad below
        auto seed_row = [&](float (&c)[D]) {
#pragma unroll
            for (int k = 0; k < D; ++k) c[k] = *reinterpret_cast<const volatile float *>(&s_c[k]);
        };
        // A point's row is only fetched when the new seed can lower its distance: the reverse triangle
        // inequality gives d >= (|p| - |c|)^2, and yakmo's float evaluation of d stays within a few ulps of
        // (cn + pn) of the true value; the margins below cover both, so `up[j] > d` is false for every skipped
        // point and the result is the reference's.  This removes ~95% of the row traffic (32 of 40 bytes/point).
        const float scn = sqrtf(cn);
        const float mrg = 4e-6f;
        if (i == 0) {
            for (int j = tid; j < N; j += blockDim.x) {
                float p[D], c[D];
                gsc_load_row<D>(Xf, j, p);
                seed_row(c);
                upf[j] = gsc_yakmo_dist<D>(p, pn[j], c, cn);
                sidf[j] = 0;
            }
        } else {
            // 4 consecutive points per thread and step: two 128-bit loads (norms, current distances) decide
            const bool al = ((reinterpret_cast<unsigned long long>(pn) | reinterpret_cast<unsigned long long>(upf)) & 15ull) == 0ull;
            const int N4 = al ? (N & ~3) : 0;
            // the loads of the next quad are issued before this one is processed (the stores to up[] below would
            // otherwise keep the compiler from overlapping them; a thread only ever touches its own quads)
            const int st4 = blockDim.x * 4;
            float4 pqn = make_float4(0.f, 0.f, 0.f, 0.f), uqn = pqn;
            if (tid * 4 < N4) { pqn = *reinterpret_cast<const float4 *>(pn + tid * 4); uqn = *reinterpret_cast<const float4 *>(upf + tid * 4); }
            for (int j4 = tid * 4; j4 < N4; j4 += st4) {
                const float4 pq = pqn, uq = uqn;
                if (j4 + st4 < N4) { pqn = *reinterpret_cast<const float4 *>(pn + j4 + st4); uqn = *reinterpret_cast<const float4 *>(upf + j4 + st4); }
                const float pjs[4] = {pq.x, pq.y, pq.z, pq.w}, ujs[4] = {uq.x, uq.y, uq.z, uq.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float t = sqrtf(pjs[q]) - scn;
                    const float lb = t * t * (1.0f - mrg) - mrg * (cn + pjs[q]) - 1e-37f;
                    if (!(lb > ujs[q])) {          // the seed may lower this distance: fetch the row
                        float p[D], c[D];
                        gsc_load_row<D>(Xf, j4 + q, p);
                        seed_row(c);
                        const float d = gsc_yakmo_dist<D>(p, pjs[q], c, cn);
                        if (ujs[q] > d) { upf[j4 + q] = d; sidf[j4 + q] = i; }
                    }
                }
            }
            for (int j = N4 + tid; j < N; j += blockDim.x) {
                const float pj = pn[j], uj = upf[j];
                const float t = sqrtf(pj) - scn;
                const float lb = t * t * (1.0f - mrg) - mrg * (cn + pj) - 1e-37f;
                if (lb > uj) continue;
                float p[D], c[D];
                gsc_load_row<D>(Xf, j, p);
                seed_row(c);
                const float d = gsc_yakmo_dist<D>(p, pj, c, cn);
                if (uj > d) { upf[j] = d; sidf[j] = i; }
            }
        }
        __syncthreads();
        if (tid == 0) { const unsigned long long t1 = clock64(); c_dist += t1 - c_t; c_t = t1; }
        if (i < K - 1 && init_type == 1) {
            // obj := 0; for j: obj += up[j]; r[j] := obj   (the reference's sequential float chain)
            if (!serial_scan) {
                const float tot = gsc_seq_prefix(upf, rf, N, s_scan);
                if (tid == 0) s_obj = tot;
            } else if (tid < 32) {
                float run = 0.0f;
                for (int base = 0; base < N; base += 32) {
                    const int j = base + tid;
                    const float v = (j < N) ? upf[j] : 0.0f;
                    float mine = 0.0f;
                    const int lim = min(32, N - base);
                    for (int l = 0; l < lim; ++l) {
                        float vv = __shfl_sync(0xffffffffu, v, l);
                        run = run + vv;
                        if (tid == l) mine = run;
                    }
                    if (j < N) rf[j] = mine;
                }
                if (tid == 0) s_obj = run;
            }
        }
        __syncthreads();
        if (tid == 0) { const unsigned long long t1 = clock64(); c_scan += t1 - c_t; c_t = t1; }
    }
    if (tid == 0 && sdbg) { unsigned long long *o = sdbg + (long long)f.slot * 4; o[0] = c_pick; o[1] = c_dist; o[2] = c_scan; o[3] = K > 0 ? (unsigned long long)K : 1ull; }
}

// ---------------------------------------------------------------------------
// K5  owner sums: per-cluster sums in POINT ORDER (the reference's summation
// order), used three ways:
//   MODE 0  float sums of feature rows, labels = seed cells   (yakmo init, last seed)
//   MODE 1  float sums of feature rows, labels = assignment   (Lloyd update)
//   MODE 2  double sums of canonicalised raw chunks           (enc:845-864)
// Thread t of block b owns cluster c = b*blockDim + t and scans all labels of
// the frame from shared-memory tiles; it accumulates only its own members, so
// each cluster's sum is formed in ascending j.  O(K*N) compares like the
// reference's own scan, but they are 1-instruction compares.
// grid = (ceil(Kmax/256), F), block 256.
// ---------------------------------------------------------------------------
#define GSC_OWNER_THREADS 256
#define GSC_OWNER_TILE 2048

template <int D>
__global__ void __launch_bounds__(GSC_OWNER_THREADS) k_owner_sums_f(const GscFrame *__restrict__ frames,
                                                                    const float *__restrict__ X,
                                                                    const int *__restrict__ labels,
                                                                    float *__restrict__ sums,   // [F][Kmax][D]
                                                                    int *__restrict__ counts,   // [F][Kmax]
                                                                    int Kmax) {
    __shared__ int s_lab[GSC_OWNER_TILE];
    const GscFrame f = frames[blockIdx.y];
    if (f.K <= 0) return;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x * blockDim.x >= f.K) return;
    const float *Xf = X + f.chunk_off * D;
    const int *lab = labels + f.chunk_off;
    float acc[D];
#pragma unroll
    for (int k = 0; k < D; ++k) acc[k] = 0.0f;
    int cnt = 0;
    for (int base = 0; base < f.N; base += GSC_OWNER_TILE) {
        const int lim = min(GSC_OWNER_TILE, f.N - base);
        __syncthreads();
        for (int t = threadIdx.x; t < lim; t += blockDim.x) s_lab[t] = lab[base + t];
        __syncthreads();
        for (int t = 0; t < lim; ++t) {
            if (s_lab[t] == c) {
                float p[D];
                gsc_load_row<D>(Xf, base + t, p);
#pragma unroll
                for (int k = 0; k < D; ++k) acc[k] = acc[k] + p[k];
                ++cnt;
            }
        }
    }
    if (c < f.K) {
        float *o = sums + ((long long)f.slot * Kmax + c) * D;
#pragma unroll
        for (int k = 0; k < D; ++k) o[k] = acc[k];
        counts[(long long)f.slot * Kmax + c] = cnt;
    }
}

// ---------------------------------------------------------------------------
// Members of every cluster in ascending point order, in O(N): one warp per frame.
//   pass 1  counts per label (shared-memory histogram)
//   pass 2  exclusive scan -> offs[0..K]
//   pass 3  STABLE scatter, 32 points at a time: __match_any_sync groups the lanes with the same label, a lane's rank
//           inside its group is the number of lower lanes in it, the group's lowest lane advances the label's
//           cursor -- groups are taken in point order and lanes in lane order, so every cluster's members come out
//           in ascending j, the order in which the reference sums them (enc:845-864, yakmo's last init step).
// The per-cluster sums that used to scan all N labels per cluster (O(K*N)) walk these lists instead.
// grid = F, block = 32, dynamic smem = 4 * (K + 1) bytes.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_group_labels(const GscFrame *__restrict__ frames, const int *__restrict__ labels,
                                                     int *__restrict__ members,   // [sumN] point indices grouped by label
                                                     int *__restrict__ offs,      // [F][Kmax+1]
                                                     int Kmax) {
    extern __shared__ int s_cur[];   // [K+1]
    constexpr unsigned FULL = 0xffffffffu;
    const GscFrame f = frames[blockIdx.x];
    const int K = f.K, N = f.N, lane = threadIdx.x;
    if (K <= 0) return;
    const int *lab = labels + f.chunk_off;
    int *mem = members + f.chunk_off;
    int *of = offs + (long long)f.slot * (Kmax + 1);
    for (int c = lane; c <= K; c += 32) s_cur[c] = 0;
    __syncwarp();
    for (int j = lane; j < N; j += 32) {
        const int l = lab[j];
        if (l >= 0 && l < K) atomicAdd(&s_cur[l], 1);
    }
    __syncwarp();
    // exclusive scan of the K counts: a contiguous stretch per lane, then the lanes' totals
    const int per = (K + 31) / 32, c0 = lane * per, c1 = min(K, c0 + per);
    int tot = 0;
    for (int c = c0; c < c1; ++c) tot += s_cur[c];
    int incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
    int run = incl - tot;
    for (int c = c0; c < c1; ++c) { const int n = s_cur[c]; s_cur[c] = run; of[c] = run; run += n; }
    if (lane == 31) { s_cur[K] = incl; of[K] = incl; }
    __syncwarp();
    for (int base = 0; base < N; base += 32) {
        const int j = base + lane;
        int l = (j < N) ? lab[j] : -1;
        if (l < 0 || l >= K) l = -1 - lane;                 // invalid / past the end: a group of its own, not stored
        const unsigned grp = __match_any_sync(FULL, l);
        const int leader = __ffs(grp) - 1, rank = __popc(grp & ((1u << lane) - 1u));
        int basep = 0;
        if (lane == leader && l >= 0) { basep = s_cur[l]; s_cur[l] = basep + __popc(grp); }
        basep = __shfl_sync(FULL, basep, leader);
        if (l >= 0) mem[basep + rank] = j;
        __syncwarp();
    }
}

// Float sums of the feature rows of every cluster's members in point order (yakmo init(): the last seed adds each
// point to its cell; Lloyd-style mean update of run()): thread per cluster over its member list.
template <int D>
__global__ void __launch_bounds__(128) k_member_sums_f(const GscFrame *__restrict__ frames, const float *__restrict__ X,
                                                       const int *__restrict__ members, const int *__restrict__ offs,
                                                       float *__restrict__ sums, int *__restrict__ counts, int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f.K) return;
    const float *Xf = X + f.chunk_off * D;
    const int *mem = members + f.chunk_off;
    const int *of = offs + (long long)f.slot * (Kmax + 1);
    const int a = of[c], b = of[c + 1];
    float acc[D];
#pragma unroll
    for (int k = 0; k < D; ++k) acc[k] = 0.0f;
    for (int t = a; t < b; ++t) {
        float p[D];
        gsc_load_row<D>(Xf, mem[t], p);
#pragma unroll
        for (int k = 0; k < D; ++k) acc[k] = acc[k] + p[k];
    }
    float *o = sums + ((long long)f.slot * Kmax + c) * D;
#pragma unroll
    for (int k = 0; k < D; ++k) o[k] = acc[k];
    counts[(long long)f.slot * Kmax + c] = b - a;
}

// centroid = sum / (float)count  (run() RVA 0x2290-0x22d3; 0/0 -> NaN kept).
// keep_empty: Lloyd variant keeps the previous centroid for empty clusters.
template <int D>
__global__ void k_means_from_sums(const GscFrame *__restrict__ frames, const float *__restrict__ sums,
                                  const int *__restrict__ counts, float *__restrict__ cen,
                                  int Kmax, int keep_empty) {
    const GscFrame f = frames[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f.K) return;
    const long long o = ((long long)f.slot * Kmax + c) * D;
    const int cnt = counts[(long long)f.slot * Kmax + c];
    if (keep_empty && cnt == 0) return;
    const float fc = (float)cnt;
#pragma unroll
    for (int k = 0; k < D; ++k) cen[o + k] = sums[o + k] / fc;
}

// Lloyd update: member rows accumulated in Double, mean rounded to Single once, so the result
// does not depend on the summation order (single GPU, or per-rank partial sums + all-reduce).
template <int D>
__global__ void __launch_bounds__(GSC_OWNER_THREADS) k_owner_sums_d(const GscFrame *__restrict__ frames,
                                                                    const float *__restrict__ X,
                                                                    const int *__restrict__ labels,
                                                                    double *__restrict__ acc,   // [F][Kmax][D+1]: D sums, count
                                                                    int Kmax) {
    __shared__ int s_lab[GSC_OWNER_TILE];
    const GscFrame f = frames[blockIdx.y];
    if (f.K <= 0) return;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x * blockDim.x >= f.K) return;
    const float *Xf = X + f.chunk_off * D;
    const int *lab = labels + f.chunk_off;
    double sum[D];
#pragma unroll
    for (int k = 0; k < D; ++k) sum[k] = 0.0;
    int cnt = 0;
    for (int base = 0; base < f.N; base += GSC_OWNER_TILE) {
        const int lim = min(GSC_OWNER_TILE, f.N - base);
        __syncthreads();
        for (int t = threadIdx.x; t < lim; t += blockDim.x) s_lab[t] = lab[base + t];
        __syncthreads();
        for (int t = 0; t < lim; ++t) {
            if (s_lab[t] == c) {
                float p[D];
                gsc_load_row<D>(Xf, base + t, p);
#pragma unroll
                for (int k = 0; k < D; ++k) sum[k] += (double)p[k];
                ++cnt;
            }
        }
    }
    if (c < f.K) {
        double *o = acc + ((long long)f.slot * Kmax + c) * (D + 1);
#pragma unroll
        for (int k = 0; k < D; ++k) o[k] = sum[k];
        o[D] = (double)cnt;
    }
}
// Same sums by scatter: one thread per point adds its row to its cluster's Double accumulators with
// red.global.add.f64 (acc zeroed beforehand).  The order of the additions is arbitrary, which is exactly what
// the Double accumulation + single rounding to Single makes harmless; ~21 points per cluster, little contention.
template <int D>
__global__ void __launch_bounds__(256) k_scatter_sums_d(const GscFrame *__restrict__ frames,
                                                        const float *__restrict__ X,
                                                        const int *__restrict__ labels,
                                                        double *__restrict__ acc,   // [F][Kmax][D+1], zeroed
                                                        int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    if (f.K <= 0) return;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= f.N) return;
    float p[D];
    gsc_load_row<D>(X + f.chunk_off * D, j, p);
    const int c = labels[f.chunk_off + j];
    double *o = acc + ((long long)f.slot * Kmax + c) * (D + 1);
#pragma unroll
    for (int k = 0; k < D; ++k) atomicAdd(o + k, (double)p[k]);
    atomicAdd(o + D, 1.0);
}

// centroid = Single(sum / count); empty clusters keep theirs.  acc may be the all-reduced buffer.
template <int D>
__global__ void k_means_from_acc(const GscFrame *__restrict__ frames, const double *__restrict__ acc,
                                 float *__restrict__ cen, int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f.K) return;
    const double *a = acc + ((long long)f.slot * Kmax + c) * (D + 1);
    const double n = a[D];
    if (!(n > 0.0)) return;
    float *o = cen + ((long long)f.slot * Kmax + c) * D;
#pragma unroll
    for (int k = 0; k < D; ++k) o[k] = (float)(a[k] / n);
}

// MODE 2: class means in the sample domain (enc:845-864), Double accumulate,
// Single store via div0.
template <int CS>
__global__ void __launch_bounds__(GSC_OWNER_THREADS) k_class_means(const GscFrame *__restrict__ frames,
                                                                   const short *__restrict__ pcm,
                                                                   const unsigned char *__restrict__ attr,
                                                                   const int *__restrict__ labels,
                                                                   float *__restrict__ means0,  // [F][Kmax][CS] cluster order
                                                                   int *__restrict__ counts,    // [F][Kmax]
                                                                   int Kmax) {
    __shared__ int s_lab[GSC_OWNER_TILE];
    const GscFrame f = frames[blockIdx.y];
    if (f.K <= 0) return;
    if (blockIdx.x * blockDim.x >= f.K) return;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int *lab = labels + f.chunk_off;
    const unsigned char *at = attr + f.chunk_off;
    double acc[CS];
#pragma unroll
    for (int k = 0; k < CS; ++k) acc[k] = 0.0;
    int cnt = 0;
    for (int base = 0; base < f.N; base += GSC_OWNER_TILE) {
        const int lim = min(GSC_OWNER_TILE, f.N - base);
        __syncthreads();
        for (int t = threadIdx.x; t < lim; t += blockDim.x) s_lab[t] = lab[base + t];
        __syncthreads();
        for (int t = 0; t < lim; ++t) {
            if (s_lab[t] == c) {
                const int n = base + t;
                const int i = n / f.C, ch = n - i * f.C;
                const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
                const unsigned char a = at[n];
                const bool rv = a & 1, ng = (a >> 1) & 1;
#pragma unroll
                for (int k = 0; k < CS; ++k) {
                    const int p = rv ? CS - 1 - k : k;
                    const double x = (i * CS + p < f.S) ? gsc_sample(row[p]) : 0.0;
                    acc[k] += x * (ng ? -1.0 : 1.0);  // enc:857
                }
                ++cnt;
            }
        }
    }
    if (c < f.K) {
        float *o = means0 + ((long long)f.slot * Kmax + c) * CS;
        const double y = (double)cnt;
#pragma unroll
        for (int k = 0; k < CS; ++k) o[k] = (float)((fabs(y) <= 1e-12) ? 0.0 : acc[k] / y);  // div0, enc:863
        counts[(long long)f.slot * Kmax + c] = cnt;
    }
}

// enc:845-864 over the member lists of k_group_labels: Double accumulate in ascending point order, Single store via div0.
template <int CS>
__global__ void __launch_bounds__(128) k_class_means_members(const GscFrame *__restrict__ frames, const short *__restrict__ pcm,
                                                             const unsigned char *__restrict__ attr,
                                                             const int *__restrict__ members, const int *__restrict__ offs,
                                                             float *__restrict__ means0, int *__restrict__ counts, int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f.K) return;
    const int *mem = members + f.chunk_off;
    const unsigned char *at = attr + f.chunk_off;
    const int *of = offs + (long long)f.slot * (Kmax + 1);
    const int a0 = of[c], b0 = of[c + 1];
    double acc[CS];
#pragma unroll
    for (int k = 0; k < CS; ++k) acc[k] = 0.0;
    for (int t = a0; t < b0; ++t) {
        const int n = mem[t];
        const int i = n / f.C, ch = n - i * f.C;
        const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
        const unsigned char a = at[n];
        const bool rv = a & 1, ng = (a >> 1) & 1;
#pragma unroll
        for (int k = 0; k < CS; ++k) {
            const int p = rv ? CS - 1 - k : k;
            const double x = (i * CS + p < f.S) ? gsc_sample(row[p]) : 0.0;
            acc[k] += x * (ng ? -1.0 : 1.0);  // enc:857
        }
    }
    float *o = means0 + ((long long)f.slot * Kmax + c) * CS;
    const double y = (double)(b0 - a0);
#pragma unroll
    for (int k = 0; k < CS; ++k) o[k] = (float)((fabs(y) <= 1e-12) ? 0.0 : acc[k] / y);  // div0, enc:863
    counts[(long long)f.slot * Kmax + c] = b0 - a0;
}

// ---------------------------------------------------------------------------
// K7  population sort + dictionary quantisation (enc:865-882), or passthrough
// dictionary (enc:891-912).  One CTA per frame; thread 0 runs the FreePascal
// quicksort (its tie order decides dictionary positions), then all threads
// quantise.  Dynamic smem: keys[Kmax] + items[Kmax] + stack[2*Kmax] ints.
// ---------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(256) k_dictionary(const GscFrame *__restrict__ frames,
                                                    const short *__restrict__ pcm, int bits,
                                                    const int *__restrict__ divider,
                                                    const float *__restrict__ means0,  // cluster order
                                                    const int *__restrict__ counts0,   // cluster order
                                                    float *__restrict__ means,         // dictionary order
                                                    int *__restrict__ order,           // [F][Kmax]
                                                    int *__restrict__ counts,          // dictionary order
                                                    short *__restrict__ dict,          // [F][Kmax][CS]
                                                    unsigned char *__restrict__ datten,
                                                    unsigned char *__restrict__ dattr,
                                                    int *__restrict__ entry,           // [sumN] or null
                                                    const int *__restrict__ labels,
                                                    int Kmax) {
    extern __shared__ int sm[];
    const GscFrame f = frames[blockIdx.x];
    const long long fo = (long long)f.slot * Kmax;
    GscLaw L;
    L.init(1.0 / (double)divider[f.slot]);
    const int obd = (1 << (bits - 1)) - 1;
    if (f.K > 0) {
        int *keys = sm, *items = sm + Kmax, *stack = sm + 2 * Kmax;
        for (int i = threadIdx.x; i < f.K; i += blockDim.x) { keys[i] = counts0[fo + i]; items[i] = i; }
        __syncthreads();
        if (threadIdx.x == 0) gsc_fpc_sort_desc(keys, items, f.K, stack);  // enc:865
        __syncthreads();
        int *inv = stack;  // reuse
        for (int i = threadIdx.x; i < f.K; i += blockDim.x) {
            const int c = items[i];
            inv[c] = i;  // enc:878
            if (order) order[fo + i] = c;
            if (counts) counts[fo + i] = keys[c];
            double x[CS];
#pragma unroll
            for (int k = 0; k < CS; ++k) {
                float m = means0[(fo + c) * CS + k];
                if (means) means[(fo + i) * CS + k] = m;
                double v = (double)m;
                x[k] = (v != v) ? 0.0 : v;  // nan0 enc:876
            }
            int a; bool ng, rv;
            gsc_chunk_attrs<CS>(x, L, a, ng, rv);  // enc:880
#pragma unroll
            for (int k = 0; k < CS; ++k) dict[(fo + i) * CS + k] = gsc_quant(x[k], obd, L.T[a], ng);  // enc:881
            datten[fo + i] = (unsigned char)a;
            if (dattr) dattr[fo + i] = (unsigned char)((ng ? 2 : 0) | (rv ? 1 : 0));
        }
        __syncthreads();
        if (entry)
            for (int j = threadIdx.x; j < f.N; j += blockDim.x)
                entry[f.chunk_off + j] = inv[labels[f.chunk_off + j]];  // enc:884-885
    } else {
        // passthrough: every chunk is its own dictionary entry (R = N <= Kmax)
        for (int n = threadIdx.x; n < f.N; n += blockDim.x) {
            const int i = n / f.C, ch = n - i * f.C;
            const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
            double x[CS];
#pragma unroll
            for (int k = 0; k < CS; ++k) x[k] = (i * CS + k < f.S) ? gsc_sample(row[k]) : 0.0;
            int a; bool ng, rv;
            gsc_chunk_attrs<CS>(x, L, a, ng, rv);
#pragma unroll
            for (int k = 0; k < CS; ++k) dict[(fo + n) * CS + k] = gsc_quant(x[k], obd, L.T[a], ng);
            datten[fo + n] = (unsigned char)a;
            if (dattr) dattr[fo + n] = (unsigned char)((ng ? 2 : 0) | (rv ? 1 : 0));
            if (entry) entry[f.chunk_off + n] = n;
        }
    }
}

// ---------------------------------------------------------------------------
// K6  KNNFit (enc:915-965): exact search over the 4R variants + epsilon band.
// Base entries V0[e][j] = Single(deq(dict[e][j], atten[e], neg=0)) live in
// shared memory (R*CS floats); the other three variants are sign / order
// images of V0 and are never materialised:
//   row e*4+0: ( V0[j])   row e*4+1: ( V0[CS-1-j])
//   row e*4+2: (-V0[j])   row e*4+3: (-V0[CS-1-j])
// (deq is odd in its sample, Single rounding is symmetric, so -V0 is exact.)
// Distance = ANN's: d=0; d += (q_j - v_j)^2 left to right, no FMA.
// Pass 1 finds dmin; the band test |sqrt(dmin/cs) - sqrt(d/cs)| <= eps is
// monotone in d, so it is turned into a threshold dthr by bisection on the
// float bit pattern; pass 2 finds the lowest row with d <= dthr and counts the
// rows inside the band.
// grid = (ceil(maxN/256), F), block 256, dyn smem = Kmax*CS*4 bytes.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool gsc_in_band(float a, float d, float fcs, float eps) {
    float b = sqrtf(d / fcs);
    return (a > b) ? ((a - b) <= eps) : ((b - a) <= eps);  // SameValue(Single)
}

// Bit j set: component j of the entry is -32768, whose sign image is itself (enc:1665-1680 negates a SmallInt with
// range checks off), so the negated variants keep +v there instead of -v.
template <int CS>
__device__ __forceinline__ unsigned gsc_min16_mask(const short *e) {
    unsigned m = 0;
#pragma unroll
    for (int j = 0; j < CS; ++j) m |= (e[j] == (short)-32768) ? (1u << j) : 0u;
    return m;
}

template <int CS>
__device__ __forceinline__ void gsc_variant_dists(const float (&q)[CS], const float (&v)[CS], unsigned m,
                                                  float &d0, float &d1, float &d2, float &d3) {
    d0 = 0.0f; d1 = 0.0f; d2 = 0.0f; d3 = 0.0f;
    if (m == 0) {
#pragma unroll
        for (int j = 0; j < CS; ++j) {
            float t0 = q[j] - v[j];
            float t1 = q[j] - v[CS - 1 - j];
            float t2 = q[j] + v[j];
            float t3 = q[j] + v[CS - 1 - j];
            float m0 = t0 * t0, m1 = t1 * t1, m2 = t2 * t2, m3 = t3 * t3;
            d0 = d0 + m0; d1 = d1 + m1; d2 = d2 + m2; d3 = d3 + m3;
        }
    } else {
#pragma unroll
        for (int j = 0; j < CS; ++j) {
            float t0 = q[j] - v[j];
            float t1 = q[j] - v[CS - 1 - j];
            float t2 = ((m >> j) & 1u) ? q[j] - v[j] : q[j] + v[j];
            float t3 = ((m >> (CS - 1 - j)) & 1u) ? q[j] - v[CS - 1 - j] : q[j] + v[CS - 1 - j];
            float m0 = t0 * t0, m1 = t1 * t1, m2 = t2 * t2, m3 = t3 * t3;
            d0 = d0 + m0; d1 = d1 + m1; d2 = d2 + m2; d3 = d3 + m3;
        }
    }
}

__device__ __forceinline__ float gsc_knnfit_epsilon(int bits, double law) {
    float maxLaw = 1.0f;  // enc:940-942 (Single accumulator, Double product)
    for (int j = 0; j <= GSC_MAX_ATT; ++j) maxLaw = (float)((double)maxLaw + (double)j * law);
    float a = 1.0f / ((float)(1 << bits) * maxLaw);  // enc:943
    double b = 1.0 / 32767.0;
    double m = ((double)a > b) ? (double)a : b;
    return (float)m;
}

template <int CS>
__global__ void __launch_bounds__(256) k_knnfit(const GscFrame *__restrict__ frames,
                                                const short *__restrict__ pcm, int bits,
                                                const int *__restrict__ divider,
                                                const short *__restrict__ dict,
                                                const unsigned char *__restrict__ datten,
                                                int *__restrict__ best,      // [sumN]
                                                int *__restrict__ use,       // [F][Kmax], zeroed
                                                int *__restrict__ band,      // [sumN] or null
                                                int *__restrict__ overfull,  // [F], zeroed
                                                int Kmax) {
    extern __shared__ float s_v[];  // [R][CS] | [R] -32768 masks (as unsigned)
    const GscFrame f = frames[blockIdx.y];
    if ((long long)blockIdx.x * blockDim.x >= f.N) return;
    const long long fo = (long long)f.slot * Kmax;
    const int R = f.R;
    unsigned *s_m = reinterpret_cast<unsigned *>(s_v + (size_t)R * CS);
    const double law = 1.0 / (double)divider[f.slot];
    GscLaw L;
    L.init(law);
    const int obd = (1 << (bits - 1)) - 1;
    for (int t = threadIdx.x; t < R * CS; t += blockDim.x) {
        const int e = t / CS;
        s_v[t] = (float)gsc_dequant(dict[fo * CS + t], obd, L.T[datten[fo + e]], false);  // enc:932
    }
    for (int e = threadIdx.x; e < R; e += blockDim.x) s_m[e] = gsc_min16_mask<CS>(dict + (fo + e) * CS);
    __syncthreads();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= f.N) return;
    const int i = n / f.C, ch = n - i * f.C;
    const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
    float q[CS];
#pragma unroll
    for (int j = 0; j < CS; ++j) q[j] = (i * CS + j < f.S) ? (float)gsc_sample(row[j]) : 0.0f;  // enc:949-950

    // pass 1: exact minimum
    float dmin = INFINITY;
    for (int e = 0; e < R; ++e) {
        float v[CS];
#pragma unroll
        for (int j = 0; j < CS; ++j) v[j] = s_v[e * CS + j];
        float d0, d1, d2, d3;
        gsc_variant_dists<CS>(q, v, s_m[e], d0, d1, d2, d3);
        dmin = fminf(dmin, fminf(fminf(d0, d1), fminf(d2, d3)));
    }
    // threshold: largest float d with in_band(d)
    const float eps = gsc_knnfit_epsilon(bits, law);
    const float fcs = (float)CS;
    const float a = sqrtf(dmin / fcs);
    unsigned lo = __float_as_uint(dmin), hi = 0x7f800000u;  // in_band(lo) true, in_band(+inf) false
    while (hi - lo > 1u) {
        unsigned mid = lo + ((hi - lo) >> 1);
        if (gsc_in_band(a, __uint_as_float(mid), fcs, eps)) lo = mid; else hi = mid;
    }
    const float dthr = __uint_as_float(lo);
    // pass 2: lowest row inside the band, and the band population
    int bi = -1, nb = 0;
    for (int e = 0; e < R; ++e) {
        float v[CS];
#pragma unroll
        for (int j = 0; j < CS; ++j) v[j] = s_v[e * CS + j];
        float d0, d1, d2, d3;
        gsc_variant_dists<CS>(q, v, s_m[e], d0, d1, d2, d3);
        const bool b0 = d0 <= dthr, b1 = d1 <= dthr, b2 = d2 <= dthr, b3 = d3 <= dthr;
        if (b0 | b1 | b2 | b3) {
            nb += (int)b0 + (int)b1 + (int)b2 + (int)b3;
            if (bi < 0) bi = e * 4 + (b0 ? 0 : b1 ? 1 : b2 ? 2 : 3);
        }
    }
    if (bi < 0) bi = 0;  // only reachable with NaN distances
    best[f.chunk_off + n] = bi;
    atomicAdd(&use[fo + (bi >> 2)], 1);  // enc:962-964
    if (band) band[f.chunk_off + n] = nb;
    if (nb > GSC_BUCKET) atomicAdd(&overfull[f.slot], 1);
}

// ---------------------------------------------------------------------------
// K6, windowed form.  The Euclidean norm is the same for the four variants of an entry (sign and order
// images), and d(q, v) >= (|q| - |v|)^2, so with the entries sorted by norm a query only has to visit the
// window of entries whose norm lies within sqrt(dmin) (pass 1) or sqrt(dthr) (pass 2) of its own -- a few
// percent of the dictionary.  k_knn_prep sorts one frame's de-quantised base variants by norm (bitonic, one
// CTA); k_knnfit_win walks outwards from the query's own norm.  Results are those of k_knnfit: the same exact
// distances, the same band threshold, the lowest ROW index inside the band (rows keep their entry numbers).
// The margin covers the float evaluation of both norms and of the exact distance.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float gsc_norm_lb(float nq, float n) {
    const float gap = fabsf(nq - n) - 1.0e-6f * (nq + n);   // both norms are within 5e-7 relative of the true ones
    return gap > 0.0f ? gap * gap * (1.0f - 2e-6f) : 0.0f;
}

template <int CS>
__global__ void __launch_bounds__(256) k_knn_prep(const GscFrame *__restrict__ frames, int bits,
                                                  const int *__restrict__ divider,
                                                  const short *__restrict__ dict,
                                                  const unsigned char *__restrict__ datten,
                                                  float *__restrict__ sV,   // [F][Kmax][CS] base variants, norm order
                                                  float *__restrict__ sN,   // [F][Kmax] norms, ascending
                                                  int *__restrict__ sE,     // [F][Kmax] entry | -32768 mask << 24
                                                  int Kmax) {
    extern __shared__ unsigned long long s_key[];   // [R2] (norm bits << 32 | entry)
    const GscFrame f = frames[blockIdx.x];
    const long long fo = (long long)f.slot * Kmax;
    const int R = f.R;
    int R2 = 1;
    while (R2 < R) R2 <<= 1;
    GscLaw L;
    L.init(1.0 / (double)divider[f.slot]);
    const int obd = (1 << (bits - 1)) - 1;
    for (int e = threadIdx.x; e < R2; e += blockDim.x) {
        unsigned long long key = ~0ull;
        if (e < R) {
            float n2 = 0.0f;
#pragma unroll
            for (int j = 0; j < CS; ++j) {
                const float v = (float)gsc_dequant(dict[(fo + e) * CS + j], obd, L.T[datten[fo + e]], false);
                n2 = fmaf(v, v, n2);
            }
            key = ((unsigned long long)__float_as_uint(sqrtf(n2)) << 32) | (unsigned)e;
        }
        s_key[e] = key;
    }
    __syncthreads();
    for (int k2 = 2; k2 <= R2; k2 <<= 1)
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < R2; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long a = s_key[i], b = s_key[l];
                    if ((a > b) == ((i & k2) == 0)) { s_key[i] = b; s_key[l] = a; }
                }
            }
            __syncthreads();
        }
    for (int p = threadIdx.x; p < R; p += blockDim.x) {
        const unsigned long long key = s_key[p];
        const int e = (int)(key & 0xffffffffu);
        sN[fo + p] = __uint_as_float((unsigned)(key >> 32));
        sE[fo + p] = e | (int)(gsc_min16_mask<CS>(dict + (fo + e) * CS) << 24);   // e < GSC_MAX_K < 2^24
#pragma unroll
        for (int j = 0; j < CS; ++j)
            sV[(fo + p) * CS + j] = (float)gsc_dequant(dict[(fo + e) * CS + j], obd, L.T[datten[fo + e]], false);   // enc:932
    }
}

template <int CS>
__global__ void __launch_bounds__(256) k_knnfit_win(const GscFrame *__restrict__ frames,
                                                    const short *__restrict__ pcm, int bits,
                                                    const int *__restrict__ divider,
                                                    const float *__restrict__ sV, const float *__restrict__ sN,
                                                    const int *__restrict__ sE,
                                                    int *__restrict__ best,      // [sumN]
                                                    int *__restrict__ use,       // [F][Kmax], zeroed
                                                    int *__restrict__ band,      // [sumN] or null
                                                    int *__restrict__ overfull,  // [F], zeroed
                                                    int Kmax) {
    extern __shared__ float s_w[];   // [R][CS] variants | [R] norms | [R] entries (as int)
    const GscFrame f = frames[blockIdx.y];
    if ((long long)blockIdx.x * blockDim.x >= f.N) return;
    const long long fo = (long long)f.slot * Kmax;
    const int R = f.R;
    float *s_v = s_w, *s_n = s_w + (size_t)R * CS;
    int *s_e = reinterpret_cast<int *>(s_n + R);
    for (int t = threadIdx.x; t < R * CS; t += blockDim.x) s_v[t] = sV[fo * CS + t];
    for (int t = threadIdx.x; t < R; t += blockDim.x) { s_n[t] = sN[fo + t]; s_e[t] = sE[fo + t]; }
    __syncthreads();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= f.N) return;
    const int i = n / f.C, ch = n - i * f.C;
    const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
    float q[CS];
    float nq2 = 0.0f;
#pragma unroll
    for (int j = 0; j < CS; ++j) { q[j] = (i * CS + j < f.S) ? (float)gsc_sample(row[j]) : 0.0f; nq2 = fmaf(q[j], q[j], nq2); }   // enc:949-950
    const float nq = sqrtf(nq2);
    // first position whose norm is >= the query's
    int lo = 0, hi = R;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_n[mid] < nq) lo = mid + 1; else hi = mid; }
    const int p0 = lo;

    // pass 1: exact minimum, walking outwards from p0 while the norm bound can still beat it
    float dmin = INFINITY;
    {
        int up = p0, dn = p0 - 1;
        bool upok = up < R, dnok = dn >= 0;
        while (upok || dnok) {
            if (upok) {
                if (gsc_norm_lb(nq, s_n[up]) > dmin) upok = false;
                else {
                    float v[CS];
#pragma unroll
                    for (int j = 0; j < CS; ++j) v[j] = s_v[up * CS + j];
                    float d0, d1, d2, d3;
                    gsc_variant_dists<CS>(q, v, (unsigned)s_e[up] >> 24, d0, d1, d2, d3);
                    dmin = fminf(dmin, fminf(fminf(d0, d1), fminf(d2, d3)));
                    upok = ++up < R;
                }
            }
            if (dnok) {
                if (gsc_norm_lb(nq, s_n[dn]) > dmin) dnok = false;
                else {
                    float v[CS];
#pragma unroll
                    for (int j = 0; j < CS; ++j) v[j] = s_v[dn * CS + j];
                    float d0, d1, d2, d3;
                    gsc_variant_dists<CS>(q, v, (unsigned)s_e[dn] >> 24, d0, d1, d2, d3);
                    dmin = fminf(dmin, fminf(fminf(d0, d1), fminf(d2, d3)));
                    dnok = --dn >= 0;
                }
            }
        }
    }
    // threshold: largest float d with in_band(d)
    const double law = 1.0 / (double)divider[f.slot];
    const float eps = gsc_knnfit_epsilon(bits, law);
    const float fcs = (float)CS;
    const float a = sqrtf(dmin / fcs);
    unsigned blo = __float_as_uint(dmin), bhi = 0x7f800000u;  // in_band(lo) true, in_band(+inf) false
    while (bhi - blo > 1u) {
        const unsigned mid = blo + ((bhi - blo) >> 1);
        if (gsc_in_band(a, __uint_as_float(mid), fcs, eps)) blo = mid; else bhi = mid;
    }
    const float dthr = __uint_as_float(blo);
    // pass 2: lowest row inside the band and the band population, same walk with the band threshold
    int bi = 0x7fffffff, nb = 0;
    for (int dir = 0; dir < 2; ++dir) {
        int p = dir ? p0 - 1 : p0;
        while (p >= 0 && p < R) {
            if (gsc_norm_lb(nq, s_n[p]) > dthr) break;
            float v[CS];
#pragma unroll
            for (int j = 0; j < CS; ++j) v[j] = s_v[p * CS + j];
            float d0, d1, d2, d3;
            gsc_variant_dists<CS>(q, v, (unsigned)s_e[p] >> 24, d0, d1, d2, d3);
            const bool b0 = d0 <= dthr, b1 = d1 <= dthr, b2 = d2 <= dthr, b3 = d3 <= dthr;
            if (b0 | b1 | b2 | b3) {
                nb += (int)b0 + (int)b1 + (int)b2 + (int)b3;
                const int r0 = (s_e[p] & 0xffffff) * 4 + (b0 ? 0 : b1 ? 1 : b2 ? 2 : 3);
                bi = min(bi, r0);
            }
            p += dir ? -1 : 1;
        }
    }
    if (bi == 0x7fffffff) bi = 0;  // only reachable with NaN distances
    best[f.chunk_off + n] = bi;
    atomicAdd(&use[fo + (bi >> 2)], 1);  // enc:962-964
    if (band) band[f.chunk_off + n] = nb;
    if (nb > GSC_BUCKET) atomicAdd(&overfull[f.slot], 1);
}

// ---------------------------------------------------------------------------
// enc:970-977: prune unused entries, sort by use count (FreePascal quicksort
// order), renumber; then emit the final dictionary and per-chunk index/attr.
// One CTA per frame.  Dynamic smem: keys[Kmax] + items[Kmax] + stack[2*Kmax].
// ---------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(256) k_finalize(const GscFrame *__restrict__ frames,
                                                  const int *__restrict__ use,
                                                  const short *__restrict__ dict,
                                                  const unsigned char *__restrict__ datten,
                                                  const int *__restrict__ best,
                                                  int *__restrict__ remap,        // [F][Kmax]
                                                  int *__restrict__ order2,       // [F][Kmax]
                                                  int *__restrict__ newR,         // [F]
                                                  short *__restrict__ out_dict,   // [F][Kmax][CS]
                                                  unsigned char *__restrict__ out_datten,
                                                  int *__restrict__ out_index,    // [sumN]
                                                  unsigned char *__restrict__ out_attr,
                                                  int Kmax) {
    extern __shared__ int sm[];
    __shared__ int s_n;
    const GscFrame f = frames[blockIdx.x];
    const long long fo = (long long)f.slot * Kmax;
    const int R = f.R;
    int *keys = sm, *items = sm + Kmax, *stack = sm + 2 * Kmax;
    for (int i = threadIdx.x; i < R; i += blockDim.x) keys[i] = use[fo + i];
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int i = 0; i < R; ++i) if (keys[i] != 0) items[n++] = i;  // Delete keeps order, enc:970-972
        gsc_fpc_sort_desc(keys, items, n, stack);                      // enc:974
        s_n = n;
    }
    __syncthreads();
    const int n = s_n;
    int *rm = stack;
    for (int i = threadIdx.x; i < R; i += blockDim.x) rm[i] = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int e = items[i];
        rm[e] = i;
        if (order2) order2[fo + i] = e;
        if (out_dict) {
#pragma unroll
            for (int k = 0; k < CS; ++k) out_dict[(fo + i) * CS + k] = dict[(fo + e) * CS + k];
            out_datten[fo + i] = datten[fo + e];
        }
    }
    __syncthreads();
    if (remap) for (int i = threadIdx.x; i < R; i += blockDim.x) remap[fo + i] = rm[i];
    if (threadIdx.x == 0 && newR) newR[f.slot] = n;
    if (best && out_index)
        for (int j = threadIdx.x; j < f.N; j += blockDim.x) {
            const int b = best[f.chunk_off + j];
            out_index[f.chunk_off + j] = rm[b >> 2];
            out_attr[f.chunk_off + j] = (unsigned char)(b & 3);
        }
}

// ---------------------------------------------------------------------------
// SURVEY.md 8(f3): the .gsc frame (TFrame.SaveStream, enc:980-1107) packed on the device, one CTA per frame.
//   header 12 B | attenuation nibbles | dictionary samples (8-bit, or 12-bit pairs in 3 bytes) |
//   u32 indexes per channel | LSB-first bit stream of per-chunk codes, flushed in 16-bit words
// A chunk's code (enc:1054-1088): Negative(1) Reversed(1) NewHeader(1) [Header(2) if its group count differs
// from the previous chunk's] then (groups+1) 3-bit groups of the index, most significant first; groups =
// floor(bsr(index)/3).  Code lengths depend on the previous chunk only, so the bit offsets are an exclusive
// prefix sum (block scan with a running carry) and every chunk ORs its bits into the zeroed output words.
// out: [F][cap] bytes, cap a multiple of 4; nbytes[F].
// ---------------------------------------------------------------------------
__device__ __forceinline__ int gsc_index_groups(int index) { return index == 0 ? 0 : (31 - __clz(index)) / 3; }

template <int CS>
__global__ void __launch_bounds__(1024) k_pack_frames(const GscFrame *__restrict__ frames, int bits, int sample_rate,
                                                      const int *__restrict__ divider, const int *__restrict__ newR,
                                                      const short *__restrict__ odict, const unsigned char *__restrict__ odatten,
                                                      const int *__restrict__ oindex, const unsigned char *__restrict__ oattr,
                                                      unsigned char *__restrict__ out, long long cap,
                                                      long long *__restrict__ nbytes, int Kmax) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const GscFrame f = frames[blockIdx.x];
    const long long fo = (long long)f.slot * Kmax;
    const int R = newR[f.slot];
    unsigned char *o = out + (long long)f.slot * cap;
    unsigned *ow = reinterpret_cast<unsigned *>(o);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // fixed-size sections
    const int att_bytes = (R + 1) / 2;
    const int smp_bytes = (bits == 8) ? R * CS : R * ((CS / 2) * 3 + (CS & 1) * 2);
    const long long head = 12 + att_bytes + smp_bytes + 4;      // bytes before the bit stream
    for (long long w = tid; w < cap / 4; w += blockDim.x) ow[w] = 0u;
    __syncthreads();
    if (tid == 0) {
        o[0] = 1; o[1] = (unsigned char)f.C;                                   // StreamVersion, ChannelCount   enc:988-989
        o[2] = (unsigned char)(R & 0xff); o[3] = (unsigned char)(R >> 8);      // ChunkCount | (BandCount-1)<<13 enc:990-991
        o[4] = (unsigned char)bits; o[5] = (unsigned char)CS;                  // enc:992-993
        o[6] = (unsigned char)(sample_rate & 0xff); o[7] = (unsigned char)((sample_rate >> 8) & 0xff);
        o[8] = (unsigned char)((sample_rate >> 16) & 0xff); o[9] = 0;          // | ChunkBlend << 24             enc:994-995
        const int dv = divider[f.slot];
        o[10] = (unsigned char)(dv & 0xff); o[11] = (unsigned char)(dv >> 8);  // enc:996-997
        const unsigned fl = (unsigned)(f.N / f.C);                             // enc:1048
        unsigned char *q = o + 12 + att_bytes + smp_bytes;
        q[0] = (unsigned char)(fl & 0xff); q[1] = (unsigned char)((fl >> 8) & 0xff);
        q[2] = (unsigned char)((fl >> 16) & 0xff); q[3] = (unsigned char)(fl >> 24);
    }
    for (int j = tid; j < att_bytes; j += blockDim.x) {                        // enc:1003-1011
        const int a0 = odatten[fo + 2 * j], a1 = (2 * j + 1 < R) ? odatten[fo + 2 * j + 1] : 0;
        o[12 + j] = (unsigned char)((a0 << 4) | a1);
    }
    unsigned char *sp = o + 12 + att_bytes;
    if (bits == 8) {                                                           // enc:1015-1018
        for (int j = tid; j < R * CS; j += blockDim.x) sp[j] = (unsigned char)((odict[fo * CS + j] + 128) & 0xff);
    } else {                                                                   // enc:1019-1039
        constexpr int per = (CS / 2) * 3 + (CS & 1) * 2;
        for (int e = tid; e < R; e += blockDim.x) {
            const short *d = odict + (fo + e) * CS;
            unsigned char *q = sp + (long long)e * per;
#pragma unroll
            for (int k = 0; k + 1 < CS; k += 2) {
                const int s1 = d[k] + 2048, s2 = d[k + 1] + 2048;
                q[(k / 2) * 3] = (unsigned char)(((s1 >> 4) & 0xf0) | ((s2 >> 8) & 0x0f));
                q[(k / 2) * 3 + 1] = (unsigned char)(s1 & 0xff);
                q[(k / 2) * 3 + 2] = (unsigned char)(s2 & 0xff);
            }
            if (CS & 1) { const int s1 = d[CS - 1] + 2048; q[(CS / 2) * 3] = (unsigned char)((s1 >> 4) & 0xf0); q[(CS / 2) * 3 + 1] = (unsigned char)(s1 & 0xff); }
        }
    }
    if (tid == 0) s_carry = 0;
    __syncthreads();   // header bytes are in place before the bit stream ORs into shared words
    const int *idx = oindex + f.chunk_off;
    const unsigned char *at = oattr + f.chunk_off;
    for (int base = 0; base < f.N; base += blockDim.x) {
        const int j = base + tid;
        unsigned code = 0;
        int len = 0;
        if (j < f.N) {
            const int ix = idx[j];
            const int g = gsc_index_groups(ix);
            const int pg = (j > 0) ? gsc_index_groups(idx[j - 1]) : -1;
            code |= (unsigned)((at[j] >> 1) & 1) << len++;     // Negative
            code |= (unsigned)(at[j] & 1) << len++;            // Reversed
            if (g == pg) { ++len; }                            // NewHeader = 0
            else { code |= 1u << len++; code |= (unsigned)g << len; len += 2; }
            for (int k = g; k >= 0; --k) { code |= (unsigned)((ix >> (3 * k)) & 7) << len; len += 3; }
        }
        // exclusive prefix sum of the code lengths inside the CTA + running carry
        long long incl = len;
#pragma unroll
        for (int of = 1; of < 32; of <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, incl, of); if (lane >= of) incl += t; }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        long long wofs = 0;
        for (int w = 0; w < warp; ++w) wofs += s_warp[w];
        const long long carry = s_carry;
        const long long bitpos = head * 8 + carry + wofs + incl - len;
        if (len > 0) {
            const unsigned long long v = (unsigned long long)code << (bitpos & 31);
            atomicOr(ow + (bitpos >> 5), (unsigned)(v & 0xffffffffu));
            if (v >> 32) atomicOr(ow + (bitpos >> 5) + 1, (unsigned)(v >> 32));
        }
        __syncthreads();
        if (tid == blockDim.x - 1) s_carry = carry + wofs + incl;
        __syncthreads();
    }
    if (tid == 0) {
        const long long nbits = s_carry;
        nbytes[f.slot] = head + 2 * ((nbits + 15) / 16);                        // flushed in 16-bit words, enc:1090-1105
    }
}

// The packed frames, each in its own `cap`-byte slot, copied back to back to their offsets in the batch's stream
// (frame order, enc:1208-1214): one CTA per frame, 16-byte loads where the destination allows.
__global__ void __launch_bounds__(256) k_compact_stream(const unsigned char *__restrict__ src, long long cap,
                                                        const long long *__restrict__ nbytes,
                                                        const long long *__restrict__ offs,
                                                        unsigned char *__restrict__ dst) {
    const long long n = nbytes[blockIdx.x];
    const unsigned char *s = src + (long long)blockIdx.x * cap;
    unsigned char *d = dst + offs[blockIdx.x];
    const long long head = min(n, (long long)((16 - (reinterpret_cast<unsigned long long>(d) & 15ull)) & 15ull));
    for (long long i = threadIdx.x; i < head; i += blockDim.x) d[i] = s[i];
    const long long body = (n - head) / 16;
    // the source of the body is not 16-byte aligned in general: assemble from 4-byte words (cap is a multiple of 4
    // and so is every frame's start; head shifts the phase by at most 15 bytes)
    for (long long i = threadIdx.x; i < body; i += blockDim.x) {
        const unsigned char *p = s + head + 16 * i;
        uint4 v;
        unsigned char *vb = reinterpret_cast<unsigned char *>(&v);
#pragma unroll
        for (int k = 0; k < 16; ++k) vb[k] = p[k];
        *reinterpret_cast<uint4 *>(d + head + 16 * i) = v;
    }
    for (long long i = head + 16 * body + threadIdx.x; i < n; i += blockDim.x) d[i] = s[i];
}

// SURVEY.md 8(f2): encoder-side reconstruction (enc:487-522, 1518-1582) and the squared error behind PsyADelta
// (enc:1862-1880).  One thread per chunk; the error sum is a sum of squared int16 differences, exact in 64-bit
// integers, so sqrt(sum / count) in Double equals the reference's sequential Double sum bit for bit.
template <int CS>
__global__ void __launch_bounds__(256) k_reconstruct(const GscFrame *__restrict__ frames, const short *__restrict__ pcm,
                                                     int bits, const int *__restrict__ divider,
                                                     const short *__restrict__ odict, const unsigned char *__restrict__ odatten,
                                                     const int *__restrict__ oindex, const unsigned char *__restrict__ oattr,
                                                     short *__restrict__ recon,              // same layout as pcm, or null
                                                     unsigned long long *__restrict__ sqerr, // [F], zeroed
                                                     int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long e2 = 0;
    if (n < f.N) {
        const long long fo = (long long)f.slot * Kmax;
        const int i = n / f.C, ch = n - i * f.C;
        const int e = oindex[f.chunk_off + n];
        const unsigned char a = oattr[f.chunk_off + n];
        const bool rv = a & 1, ng = (a >> 1) & 1;
        GscLaw L;
        L.init(1.0 / (double)divider[f.slot]);
        const int obd = (1 << (bits - 1)) - 1;
        const double coeff = L.T[odatten[fo + e]];
        const long long ro = f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
#pragma unroll
        for (int j = 0; j < CS; ++j) {
            if (i * CS + j < f.S) {
                const double smp = gsc_dequant(odict[(fo + e) * CS + (rv ? CS - 1 - j : j)], obd, coeff, ng);   // enc:510
                double r = rint(smp * 32767.0);                                                                  // enc:1638-1641
                r = r < -32768.0 ? -32768.0 : (r > 32767.0 ? 32767.0 : r);
                const int o16 = (int)r;
                if (recon) recon[ro + j] = (short)o16;
                const long long d = (long long)pcm[ro + j] - (long long)o16;
                e2 += (unsigned long long)(d * d);
            }
        }
    }
    for (int of = 16; of > 0; of >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, of);
    if ((threadIdx.x & 31) == 0 && e2) atomicAdd(&sqerr[f.slot], e2);
}

// ---------------------------------------------------------------------------
// Lloyd assign: exact nearest centroid (ANN distance, lowest index on ties).
// A cheap certified lower bound
//   lb = (|c|^2)(1-g) - 2 x.c + (|x|^2)(1-g)   <=  d_exact
// filters candidates; only rows with lb <= best are evaluated in the exact
// operation order, so the result is the exact argmin.
// grid = (ceil(maxN/(128*P)), F), block 128.
// ---------------------------------------------------------------------------
#define GSC_LB_GAMMA 7.62939453125e-06f  // 2^-17, covers every rounding of both forms (DESIGN.md)
#define GSC_ASSIGN_P 8            // points per thread (4 FFMA2 pairs)
#define GSC_ASSIGN_T 128          // threads per CTA
#define GSC_ASSIGN_TILE 512       // centroids per shared-memory tile

__device__ __forceinline__ unsigned long long gsc_a_pk2(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void gsc_a_upk2(unsigned long long v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long gsc_a_ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}

// ---- 1-D bulk copies (TMA, cp.async.bulk) + mbarrier: the codebook tiles of k_assign ----
__device__ __forceinline__ unsigned gsc_smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void gsc_mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gsc_smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void gsc_mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gsc_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gsc_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(gsc_smem_addr(dst)), "l"(src), "r"(bytes), "r"(gsc_smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void gsc_mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "GSC_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra GSC_DONE_%=;\n"
        "bra GSC_WAIT_%=;\n"
        "GSC_DONE_%=:\n"
        "}\n" ::"r"(gsc_smem_addr(bar)), "r"(parity) : "memory");
}

// h_c = -0.5 |c|^2 (1 - g) over the bound's dimensions, for every centroid of every frame (rows padded to a multiple
// of 4 per frame so that a tile of them is a legal bulk copy; the pad never wins: NaN)
template <int D>
__global__ void k_cen_h(const GscFrame *__restrict__ frames, const float *__restrict__ cen, float *__restrict__ ch, int Kmax, int Kpad) {
    constexpr int DF = (D >= 8) ? D / 2 : D;
    const GscFrame f = frames[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Kpad) return;
    float h = __int_as_float(0x7fc00000);
    if (c < f.K) {
        const float *r = cen + ((long long)f.slot * Kmax + c) * D;
        float nc = 0.0f;
#pragma unroll
        for (int k = 0; k < DF; ++k) nc = fmaf(r[k], r[k], nc);
        h = -0.5f * nc * (1.0f - GSC_LB_GAMMA);
    }
    ch[(long long)f.slot * Kpad + c] = h;
}

// Register tile: 8 points per thread held as 4 packed pairs, so one FFMA2 (fma.rn.f32x2) advances the
// lower-bound score of two points; the codebook streams through shared memory in tiles of 512 centroids (rows 16 KB
// + h 2 KB) that ONE thread requests with bulk async copies (TMA, cp.async.bulk) into a two-deep ring: the copy of
// tile t+1 is in flight while tile t is scored, its arrival is an mbarrier phase, and the only block barrier left per
// tile is the one that frees a buffer.  Tile reads are broadcast loads (2 x LDS.128 + 1 x LDS.32 per centroid for 64
// FMAs).  Per (point, centroid): 8 FMAs + 1 compare; the exact ANN-order distance is evaluated only for centroids whose
// certified lower bound does not exceed the point's current best, so the result is the exact argmin (lowest index on
// ties).
// P points per thread: 8 for batches (fewest tile reads per FMA), 2 when a launch would otherwise have fewer CTAs than
// the SMs can hold (one oversized frame split over many GPUs: a shard of 131,072 points is 128 CTAs at P = 8).
template <int D, int P>
__global__ void __launch_bounds__(GSC_ASSIGN_T) k_assign(const GscFrame *__restrict__ frames,
                                                         const float *__restrict__ X,
                                                         const float *__restrict__ cen,  // [F][Kmax][D]
                                                         const float *__restrict__ ch,   // [F][Kpad] (k_cen_h)
                                                         int *__restrict__ labels, float *__restrict__ dist,
                                                         int Kmax, int Kpad) {
    constexpr int PP = P / 2;
    // dimensions of the bound: the second half of a feature row is the 1e-5-scaled cepstrum (enc:362); dropping
    // those non-negative terms keeps lb <= d and halves the FMA work
    constexpr int DF = (D >= 8) ? D / 2 : D;
    constexpr int TILE = (D > 8) ? GSC_ASSIGN_TILE / 2 : GSC_ASSIGN_TILE;   // two buffers inside 48 KB of static shared memory
    __shared__ __align__(128) float s_c[2][TILE * D];
    __shared__ __align__(16) float s_h[2][TILE];  // -0.5*|c|^2*(1-g), NaN-safe
    __shared__ __align__(8) unsigned long long s_bar[2];
    const GscFrame f = frames[blockIdx.y];
    const int K = f.K;
    const long long base = (long long)blockIdx.x * blockDim.x * P;
    if (base >= f.N) return;
    const float *Xf = X + f.chunk_off * D;
    const float *cf = cen + (long long)f.slot * Kmax * D;
    const float *hf = ch + (long long)f.slot * Kpad;
    const int ntiles = (K + TILE - 1) / TILE;
    auto request = [&](int t) {     // one thread: arm the buffer's barrier with the byte count, start both copies
        const int k0 = t * TILE, kt = min(TILE, K - k0), buf = t & 1;
        const unsigned bc = (unsigned)kt * D * 4u, bh = (unsigned)((kt + 3) & ~3) * 4u;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the buffer's last readers (generic proxy) came first
        gsc_mbar_expect_tx(&s_bar[buf], bc + bh);
        gsc_bulk_g2s(s_c[buf], cf + (long long)k0 * D, bc, &s_bar[buf]);
        gsc_bulk_g2s(s_h[buf], hf + k0, bh, &s_bar[buf]);
    };
    if (threadIdx.x == 0) {
        gsc_mbar_init(&s_bar[0], 1); gsc_mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0 && ntiles > 0) request(0);
    float x[P][D], thr[P], bd[P], hx[P];
    int bi[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const long long j = base + (long long)p * blockDim.x + threadIdx.x;
        if (j < f.N) gsc_load_row<D>(Xf, j, x[p]);
        else {
#pragma unroll
            for (int k = 0; k < D; ++k) x[p][k] = 0.0f;
        }
        float nx = 0.0f;
#pragma unroll
        for (int k = 0; k < DF; ++k) nx = fmaf(x[p][k], x[p][k], nx);
        hx[p] = 0.5f * nx * (1.0f - GSC_LB_GAMMA) - 1e-30f;
        bd[p] = INFINITY; bi[p] = 0;
        thr[p] = -INFINITY;  // candidate iff s >= thr  (s = x.c - 0.5|c|^2(1-g))
    }
    unsigned long long xp[PP][DF];   // (x[2q][k], x[2q+1][k])
#pragma unroll
    for (int q = 0; q < PP; ++q)
#pragma unroll
        for (int k = 0; k < DF; ++k) xp[q][k] = gsc_a_pk2(x[2 * q][k], x[2 * q + 1][k]);
    for (int t = 0; t < ntiles; ++t) {
        const int k0 = t * TILE, kt = min(TILE, K - k0), buf = t & 1;
        // the other buffer was released by the barrier that ended tile t-1: refill it while this tile is scored
        if (threadIdx.x == 0 && t + 1 < ntiles) request(t + 1);
        gsc_mbar_wait(&s_bar[buf], (unsigned)((t >> 1) & 1));
        const float *sc = s_c[buf], *sh = s_h[buf];
#pragma unroll 2
        for (int c = 0; c < kt; ++c) {
            float cc[DF];
            if (DF % 4 == 0) {
#pragma unroll
                for (int k = 0; k < DF / 4; ++k) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(&sc[c * D + 4 * k]);
                    cc[4 * k] = t4.x; cc[4 * k + 1] = t4.y; cc[4 * k + 2] = t4.z; cc[4 * k + 3] = t4.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < DF; ++k) cc[k] = sc[c * D + k];
            }
            const float h = sh[c];
            unsigned long long s2[PP];
#pragma unroll
            for (int q = 0; q < PP; ++q) s2[q] = gsc_a_pk2(h, h);
#pragma unroll
            for (int k = 0; k < DF; ++k) {
                const unsigned long long ck = gsc_a_pk2(cc[k], cc[k]);
#pragma unroll
                for (int q = 0; q < PP; ++q) s2[q] = gsc_a_ffma2(xp[q][k], ck, s2[q]);
            }
            float sv[P];
#pragma unroll
            for (int q = 0; q < PP; ++q) gsc_a_upk2(s2[q], sv[2 * q], sv[2 * q + 1]);
            bool any = false;
#pragma unroll
            for (int p = 0; p < P; ++p) any |= (sv[p] >= thr[p]);
            if (any) {
#pragma unroll
                for (int p = 0; p < P; ++p)
                    if (sv[p] >= thr[p]) {
                        float cr[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) cr[k] = sc[c * D + k];
                        const float d = gsc_ann_dist<D>(x[p], cr);
                        if (d < bd[p]) {
                            bd[p] = d; bi[p] = k0 + c;
                            // lb <= d  <=>  hx - s <= d/2  <=>  s >= hx - d/2
                            thr[p] = hx[p] - 0.5f * d;
                        }
                    }
            }
        }
        __syncthreads();    // everybody is done with this buffer: it may be refilled (tile t+2)
    }
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const long long j = base + (long long)p * blockDim.x + threadIdx.x;
        if (j < f.N) {
            labels[f.chunk_off + j] = bi[p];
            if (dist) dist[f.chunk_off + j] = bd[p];
        }
    }
}

// yakmo reassignment (run() after the mean update): nearest centroid under the
// norm-expansion distance, earliest centroid on ties.  Simple exact form.
template <int D>
__global__ void __launch_bounds__(128) k_assign_yakmo(const GscFrame *__restrict__ frames,
                                                      const float *__restrict__ X,
                                                      const float *__restrict__ pnorm,
                                                      const float *__restrict__ cen,
                                                      int *__restrict__ labels, int Kmax) {
    __shared__ float s_c[GSC_ASSIGN_TILE * D];
    __shared__ float s_n[GSC_ASSIGN_TILE];
    const GscFrame f = frames[blockIdx.y];
    const int K = f.K;
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if ((long long)blockIdx.x * blockDim.x >= f.N) return;
    const float *cf = cen + (long long)f.slot * Kmax * D;
    float x[D];
    float pn = 0.0f;
    int bi = 0;
    if (j < f.N) {
        gsc_load_row<D>(X + f.chunk_off * D, j, x);
        pn = pnorm[f.chunk_off + j];
        bi = labels[f.chunk_off + j];
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) x[k] = 0.0f;
    }
    float bd = INFINITY;
    for (int k0 = 0; k0 < K; k0 += GSC_ASSIGN_TILE) {
        const int kt = min(GSC_ASSIGN_TILE, K - k0);
        __syncthreads();
        for (int t = threadIdx.x; t < kt * D; t += blockDim.x) s_c[t] = cf[(long long)k0 * D + t];
        __syncthreads();
        for (int t = threadIdx.x; t < kt; t += blockDim.x) {
            float nrm = 0.0f;  // run(): norm += v*v in k order
#pragma unroll
            for (int k = 0; k < D; ++k) { float m = s_c[t * D + k] * s_c[t * D + k]; nrm = m + nrm; }
            s_n[t] = nrm;
        }
        __syncthreads();
        for (int c = 0; c < kt; ++c) {
            float cc[D];
#pragma unroll
            for (int k = 0; k < D; ++k) cc[k] = s_c[c * D + k];
            float d = gsc_yakmo_dist<D>(x, pn, cc, s_n[c]);
            if (d < bd) { bd = d; bi = k0 + c; }
        }
    }
    if (j < f.N) labels[f.chunk_off + j] = bi;
}

// ---------------------------------------------------------------------------
// Legacy ANN ABI (ext:118-123): exact brute-force k-NN of ONE query against n
// points of runtime dimension dd.  One CTA; distances go to scratch, then the
// cnt smallest by (distance, index) are extracted in ascending order.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_ann_query(const float *__restrict__ pts, int n, int dd,
                                                   const float *__restrict__ q, int cnt,
                                                   float *__restrict__ scratch,  // [n]
                                                   int *__restrict__ idxs, float *__restrict__ errs) {
    __shared__ unsigned long long s_best[8];
    __shared__ unsigned long long s_pick;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float d = 0.0f;
        for (int k = 0; k < dd; ++k) {
            float t = q[k] - pts[(long long)i * dd + k];
            float m = t * t;
            d = d + m;
        }
        scratch[i] = d;
    }
    __syncthreads();
    for (int r = 0; r < cnt; ++r) {
        unsigned long long mine = ~0ull;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            float d = scratch[i];
            if (d == d && d >= 0.0f) {  // taken rows are marked with -1
                unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)i;
                mine = key < mine ? key : mine;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long other = __shfl_xor_sync(0xffffffffu, mine, o);
            mine = other < mine ? other : mine;
        }
        if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = mine;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = s_best[0];
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) b = s_best[w] < b ? s_best[w] : b;
            s_pick = b;
            if (b != ~0ull) {
                idxs[r] = (int)(unsigned)(b & 0xffffffffu);
                errs[r] = __uint_as_float((unsigned)(b >> 32));
                scratch[(unsigned)(b & 0xffffffffu)] = -1.0f;
            } else {
                idxs[r] = -1;
                errs[r] = INFINITY;
            }
        }
        __syncthreads();
    }
}

// gsc_log_cr over an array (gsc_log_array: lets a host check the library's logarithm value by value).
__global__ void k_log_array(const double *__restrict__ x, double *__restrict__ y, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = gsc_log_cr(x[i]);
}

// FP32 FFMA throughput probe (roofline denominator, SURVEY.md 8d).
__global__ void __launch_bounds__(256) k_ffma_probe(float *out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
    float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float b = 0.999f, c = 1e-3f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
            a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
