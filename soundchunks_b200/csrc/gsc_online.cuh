// gsc_online.cuh -- K4/K5: the reference's online k-means (enc:699-765
// TFrame.KNNScanReduce), one point at a time against the LIVE centroids.
//
// The rule is sequential in the points (each update moves one centroid before
// the next query).  The kernel reproduces that sequence bit for bit while
// working on 32 points at a time: ONE CTA PER FRAME, the frames of a batch run
// side by side on the SMs.
//
// Per point (arithmetic of the result is the reference's, bit for bit):
//   best  := argmin_c  d(x, c),  d = sum_k (x_k - c_k)^2   float, left to
//            right, no FMA (ANN annkSearch, eps = 0; lowest index on ties)
//   rate  := Single(1 / sqrt(cnt_prev[best]))               enc:735
//   c_best += (x - c_best) * rate                            enc:736-740
//   err   += sqrt(d / D)   (Single sqrt, Double accumulate)  enc:743
//
// Data placement (K = 4096, D = 8):
//   shared memory  exact centroid rows K x 8 fp32 = 128 KB (the truth; read for
//                  exact scoring, updates and the broadcast filter), h_c 16 KB,
//                  per-centroid rate 16 KB, counts 16 KB, moved flags 4 KB,
//                  point tile 8 KB, candidate lists 8 KB, survivor queues 8 KB
//   registers      FILTER copy: first DF = 4 dims of the thread's CPT = 16
//                  centroids (64 regs) + h_c = -0.5|c|^2(1-g) (16 regs)
//   HBM            one 32-byte row per point per pass (streamed through smem)
//
// Codebook order: the kernel works on a copy sorted by c0 (first feature,
// re-sorted at the start of every pass); a CELL is CPT consecutive slots and
// belongs to one thread, consecutive cells to different warps.  A point visits
// only the cells whose exact c0 range meets [x0 - sqrt(U), x0 + sqrt(U)].
//
// Schedule: points are taken in batches of B = 32 (lane b of warp 0 = point b).
//  Phase 1 (all warps, codebook frozen at the batch start S0).  For every
//    (cell, point) pair that passes the slab test the first DF dimensions give
//        s_c = x.c + h_c                          (DF FMAs per centroid)
//    which certifies the LOWER bound
//        lb_c = |x|^2(1-g) - 2 s_c <= sum_{k<DF}(x_k-c_k)^2 <= d(x,c)
//    (dropped squared terms are >= 0 and tiny -- the 1e-5-scaled cepstral
//    features, enc:362; g = 2^-17 covers every rounding of both forms).
//    U_b is the exact distance to the centroid the point chose in the previous
//    pass (its seed cell in pass 0).  Neighbouring points have neighbouring c0,
//    so a batch hits a few cells with most of its points: cells with many points
//    are evaluated by the whole warp (lane = point, the cell's rows broadcast
//    from shared memory), the others by their owner from the register copy with
//    FFMA2, two points per trip; a cost model picks the split per warp and batch.
//    Centroids with lb_c <= U_b go to the warp's survivor queue; at the end of
//    the phase the queue is scored densely, one survivor per lane, in the exact
//    operation order, and the (d bits << 32 | index) keys are appended to the
//    points' candidate lists.
//  Phase 2 (warp 0) resolves the batch in ROUNDS.  In a round every unresolved
//    lane t proposes the minimum of (a) its best list key among centroids not
//    moved since S0 and (b) its best fresh key among centroids moved in this
//    batch.  The proposal is CERTIFIED iff d_win <= U_t and the list did not
//    overflow: every unmoved centroid with d <= d_win has lb <= U_t and is on
//    the list, every moved one was scored fresh, so the key minimum is the
//    exact argmin with the lowest index on ties.  All proposing lanes compute
//    their updated rows speculatively; lane t then scores the rows of lanes
//    u < t and is in CONFLICT if one of them is its own winner or beats it.
//    Lanes before the first conflicting / uncertified lane are exactly what
//    the sequential rule produces (by induction: nothing before them touches
//    their winner or offers a closer row) and commit together; the rest go to
//    the next round with the fresh keys they just computed.  The pair scoring
//    of a round is spread over all warps (warp w takes the rows u = t0+w,
//    t0+w+W, ...), warp 0 proposes and commits.  An uncertified lane at the
//    head of a round is resolved by RE-FILTERING that one point with the whole
//    CTA against its best known exact distance (always a valid bound; -inf
//    threshold = exhaustive scan when nothing is known), inside the same batch.
// Shared memory is addressed through an opaque 32-bit base (inline ld/st.shared)
// so the shared-window base is not rematerialised (S2UR SR_CgaCtaId) in loops.
#pragma once
#include "gsc_device.cuh"

#define GSC_ON_TP 256         // points per shared-memory tile
#define GSC_ON_B 32           // points per batch (one per lane of the resolving warp)
#define GSC_ON_L 32           // candidate list capacity per point
#define GSC_ON_G 7.62939453125e-06f   // 2^-17
#define GSC_NONE 0xffffffffu
#define GSC_KNONE 0xffffffffffffffffull
#define GSC_MODE_DONE 0
#define GSC_MODE_REFILTER 1
#define GSC_MODE_SCAN 2

// ---- shared-memory access through an opaque 32-bit address -------------------
__device__ __forceinline__ unsigned gsc_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned gsc_opaque(unsigned v) { unsigned r; asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v)); return r; }
__device__ __forceinline__ float gsc_lds_f(unsigned a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ int gsc_lds_i(unsigned a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ unsigned long long gsc_lds_u64(unsigned a) { unsigned long long v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ double gsc_lds_d(unsigned a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ float4 gsc_lds_f4(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void gsc_sts_f(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void gsc_sts_i(unsigned a, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void gsc_sts_u64(unsigned a, unsigned long long v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void gsc_sts_d(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void gsc_sts_f4(unsigned a, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void gsc_atoms_or(unsigned a, unsigned v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void gsc_atoms_min_u64(unsigned a, unsigned long long v) { asm volatile("red.shared.min.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ int gsc_atoms_add(unsigned a, int v) { int o; asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o; }

__device__ __forceinline__ int gsc_lds_u8(unsigned a) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return (int)v; }
__device__ __forceinline__ void gsc_sts_u8(unsigned a, int v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

template <int D>
__device__ __forceinline__ void gsc_lds_row(unsigned a, float (&r)[D]) {
    if (D % 4 == 0) {
#pragma unroll
        for (int k = 0; k < D / 4; ++k) {
            const float4 t = gsc_lds_f4(a + 16u * k);
            r[4 * k] = t.x; r[4 * k + 1] = t.y; r[4 * k + 2] = t.z; r[4 * k + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) r[k] = gsc_lds_f(a + 4u * k);
    }
}
template <int D>
__device__ __forceinline__ void gsc_sts_row(unsigned a, const float (&r)[D]) {
    if (D % 4 == 0) {
#pragma unroll
        for (int k = 0; k < D / 4; ++k) gsc_sts_f4(a + 16u * k, make_float4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]));
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) gsc_sts_f(a + 4u * k, r[k]);
    }
}

__device__ __forceinline__ unsigned long long gsc_pack(unsigned dbits, unsigned idx) {
    return ((unsigned long long)dbits << 32) | idx;
}
__device__ __forceinline__ unsigned gsc_kd(unsigned long long k) { return (unsigned)(k >> 32); }
__device__ __forceinline__ unsigned gsc_ki(unsigned long long k) { return (unsigned)(k & 0xffffffffu); }
// The low word of a key is (original centroid index << 16) | slot: ties in the distance are broken by the
// ORIGINAL index (the reference's order), the slot (position in the kernel's c0-sorted codebook) addresses memory.
__device__ __forceinline__ unsigned gsc_ks(unsigned long long k) { return (unsigned)(k & 0xffffu); }
__device__ __forceinline__ int gsc_lds_u16(unsigned a) { unsigned v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return (int)v; }
__device__ __forceinline__ void gsc_sts_u16(unsigned a, int v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ float gsc_rate(int cnt) {  // enc:735
    return (float)(1.0 / sqrt((double)cnt));
}

// ---- packed FP32 pairs: one FFMA2 (fma.rn.f32x2, sm_100) does the filter FMA of two centroids ----
__device__ __forceinline__ unsigned long long gsc_pk2(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void gsc_upk2(unsigned long long v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long gsc_ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}
// s[2p], s[2p+1] = x . c + h for the thread's CPT centroids (DF = 4 filter dimensions)
template <int CPT, int DF>
__device__ __forceinline__ void gsc_filter_scores(const float (&x)[DF], const unsigned long long (&fcp)[CPT / 2][DF],
                                                  const unsigned long long (&hp)[CPT / 2], float (&s)[CPT]) {
    unsigned long long xx[DF], sp[CPT / 2];
#pragma unroll
    for (int k = 0; k < DF; ++k) xx[k] = gsc_pk2(x[k], x[k]);
#pragma unroll
    for (int p = 0; p < CPT / 2; ++p) sp[p] = hp[p];
#pragma unroll
    for (int k = 0; k < DF; ++k)
#pragma unroll
        for (int p = 0; p < CPT / 2; ++p) sp[p] = gsc_ffma2(xx[k], fcp[p][k], sp[p]);
#pragma unroll
    for (int p = 0; p < CPT / 2; ++p) gsc_upk2(sp[p], s[2 * p], s[2 * p + 1]);
}
// replace centroid j (compile-time) of the packed filter copy
template <int CPT, int DF>
__device__ __forceinline__ void gsc_filter_set(unsigned long long (&fcp)[CPT / 2][DF], unsigned long long (&hp)[CPT / 2], int j,
                                               const float *r, float hv) {
#pragma unroll
    for (int p = 0; p < CPT / 2; ++p) {
        if (j == 2 * p || j == 2 * p + 1) {
#pragma unroll
            for (int k = 0; k < DF; ++k) {
                float lo, hi;
                gsc_upk2(fcp[p][k], lo, hi);
                fcp[p][k] = (j == 2 * p) ? gsc_pk2(r[k], hi) : gsc_pk2(lo, r[k]);
            }
            float lo, hi;
            gsc_upk2(hp[p], lo, hi);
            hp[p] = (j == 2 * p) ? gsc_pk2(hv, hi) : gsc_pk2(lo, hv);
        }
    }
}

// minimum of 64-bit keys over a warp (two 32-bit redux steps)
__device__ __forceinline__ unsigned long long gsc_warp_min_key(unsigned long long k) {
    const unsigned kd = gsc_kd(k), ki = gsc_ki(k);
    const unsigned m = __reduce_min_sync(0xffffffffu, kd);
    const unsigned mi = __reduce_min_sync(0xffffffffu, kd == m ? ki : GSC_NONE);
    return gsc_pack(m, mi);
}

// shared-memory layout (byte offsets from the base)
template <int D, int CPT, int T>
struct GscOnLayout {
    static constexpr int KP = T * CPT;
    static constexpr unsigned X = 0;                                  // float [TP][D]
    static constexpr unsigned HX = X + GSC_ON_TP * D * 4;             // float [TP]
    static constexpr unsigned G = HX + GSC_ON_TP * 4;                 // int   [TP]
    static constexpr unsigned LIST = G + GSC_ON_TP * 4;               // u64   [L][B] (slot-major)
    static constexpr unsigned LISTN = LIST + GSC_ON_B * GSC_ON_L * 8; // int   [B] entries per point (may exceed L: overflow)
    // thresholds and slabs of the batch: every warp computes the same 32 values and keeps its OWN copy (written
    // and read behind the warp's own __syncwarp, no block barrier and no cross-warp sharing)
    static constexpr unsigned THRW = LISTN + GSC_ON_B * 4;            // float [W][B] candidate thresholds
    static constexpr unsigned XLO = THRW + (T / 32) * GSC_ON_B * 4;   // float [W][B] slab x0 - r
    static constexpr unsigned XHI = XLO + (T / 32) * GSC_ON_B * 4;    // float [W][B] slab x0 + r
    static constexpr unsigned MOVED = XHI + (T / 32) * GSC_ON_B * 4;  // int   [B] distinct centroids moved in this batch
    static constexpr unsigned ROWS = MOVED + GSC_ON_B * 4;            // float [B][D]
    static constexpr unsigned WS = ROWS + GSC_ON_B * D * 4;           // int   [B]
    static constexpr unsigned ETB = WS + GSC_ON_B * 4;                // float [2][B] distances of the committed points
    static constexpr unsigned WKEY = ETB + 2 * GSC_ON_B * 4;          // u64   [B][W] re-filter minima per (request, warp)
    // u64 [W][UW][B(lane)] fresh keys of a round as running minima: warp w scores rows u = t0+w+i*W (i < UW = B/W
    // rounded up), entry [w][i][lane] is the minimum over the first i+1 of them (W * UW * B * 8 = 8 KB for W = 2, 4, 8)
    static constexpr unsigned FK = WKEY + GSC_ON_B * (T / 32) * 8;
    static constexpr unsigned KEYS = FK + GSC_ON_B * GSC_ON_B * 8;    // u64   [B] proposals of a round
    static constexpr unsigned ABEST = KEYS + GSC_ON_B * 8;            // u64   [B] best key of each point's stored list entries
    static constexpr unsigned CB = ABEST + GSC_ON_B * 8;              // u32   [B] conflict ballots per row u
    static constexpr unsigned DIRTY = CB + GSC_ON_B * 4;              // u32   [T] moved centroids per owner thread
    static constexpr unsigned EPTS = DIRTY + T * 4;                   // int   [B] points to re-filter
    static constexpr unsigned ETHRS = EPTS + GSC_ON_B * 4;            // float [B] ... and their thresholds
    static constexpr unsigned T0 = ETHRS + GSC_ON_B * 4;              // int
    static constexpr unsigned SLOT0 = T0 + 4;                         // int   slot of original centroid 0
    static constexpr unsigned NE = SLOT0 + 4;                         // int
    static constexpr unsigned MODE = NE + 4;                          // int
    static constexpr unsigned STOP = MODE + 4;                        // int
    static constexpr unsigned ERR = ((STOP + 4 + 7) / 8) * 8;         // double
    static constexpr unsigned S2O = ((ERR + 8 + 15) / 16) * 16;       // u16   [KP] slot -> original centroid index
    static constexpr unsigned MFLAG = ((S2O + 2 * KP + 15) / 16) * 16; // u8    [KP]
    static constexpr unsigned RATE = ((MFLAG + KP + 15) / 16) * 16;   // float [KP]
    static constexpr unsigned CNT = RATE + KP * 4;                    // int   [KP] hits of the running pass (+1), enc:717-721, 744, 754-758
    static constexpr unsigned H = ((CNT + KP * 4 + 15) / 16) * 16;    // float [KP] h_c = -0.5|c|^2(1-g) over the filter dimensions
    static constexpr unsigned C = H + KP * 4;                         // float [KP][D]
    static constexpr unsigned TOTAL = C + KP * D * 4;
    static_assert(TOTAL <= 227 * 1024, "shared memory budget of one SM");
};

// GSC_ONLINE_CHECKS (debug builds of tools/spill_probe.py only; compute-sanitizer is not available on the GPU pool):
// bounds of every shared-memory index the kernel forms, and the invariants of its cross-warp hand-offs (register
// filter copy == shared rows unless flagged dirty, empty candidate lists / clear moved flags at a batch start).
// Failures are counted in the launch's debug buffer (slot 8: count, slot 9: first failing source line).
#ifdef GSC_ONLINE_CHECKS
#define GSC_CHK(cond) do { if (!(cond) && chk) { atomicAdd(chk, 1ull); atomicCAS(chk + 1, 0ull, (unsigned long long)__LINE__); } } while (0)
#else
#define GSC_CHK(cond) ((void)0)
#endif
// GSC_ONLINE_TIMING (timing builds of tools/online_serial.py only): warp 0 takes clock() at the borders of its
// sections and thread 0 adds the cycles of each, per pass, to the launch's debug buffer (slots 10..15):
//   10 (a) bar 1 -> first bar 2: batch open + the first round's proposals      11 (b) R3 commit
//   12 (c) R3 take-over of fresh keys, moved checks, list re-scans               13 (d) R3' + R1 of the later rounds
//   14 (e) bar 2 -> bar 3: R2 (all warps) and both barriers                       15 (f) the whole batch
// (a)..(d) are the sections in which warp 0 alone issues while the other warps wait at bar 2.
#ifdef GSC_ONLINE_TIMING
#define GSC_TM(i) do { const unsigned tm_n = (unsigned)clock(); tm_acc[i] += tm_n - tm_t; tm_t = tm_n; } while (0)
#else
#define GSC_TM(i) ((void)0)
#endif
// GSC_ONLINE_MAXNREG (debug builds of tools/spill_probe.py only): cap the registers below what the kernel needs, so
// that ptxas spills -- the results must not change.
#ifdef GSC_ONLINE_MAXNREG
#define GSC_ONLINE_BOUNDS(T) __maxnreg__(GSC_ONLINE_MAXNREG)
#else
#define GSC_ONLINE_BOUNDS(T) __launch_bounds__(T)
#endif
template <int D, int CPT, int T>
__global__ void GSC_ONLINE_BOUNDS(T) k_online(const GscFrame *__restrict__ frames,
                                              const float *__restrict__ X,       // [sumN][D]
                                              float *__restrict__ cen,           // [F][Kmax][D] in/out
                                              int *__restrict__ labels,          // [sumN] in: guesses, out: labels
                                              int *__restrict__ passes_out,      // [F]
                                              double *__restrict__ err_out,      // [F]
                                              double tol, int max_passes, int Kmax, int force_exact, float slack,
                                              unsigned long long *__restrict__ dbg,
                                              // a launch runs at most `slice_passes` passes of every unfinished frame; the
                                              // frame's state between launches is its centroids, labels, pass count,
                                              // error sum and the hit counts of its last pass (original centroid order)
                                              int slice_passes, int *__restrict__ cnt_state, int *__restrict__ done) {
    using Ly = GscOnLayout<D, CPT, T>;
    static_assert(T >= 64, "thread 32 accumulates the error sum");
    constexpr int DF = (D >= 8) ? D / 2 : D;   // filter dimensions
    constexpr int W = T / 32;
    constexpr int KP = T * CPT;
    constexpr int B = GSC_ON_B, L = GSC_ON_L;
    constexpr int UW = (B + W - 1) / W;        // rows a warp scores in a round of R2
    static_assert(W * UW * B <= B * B, "running minima of the fresh keys fit the FK region");
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smraw[];
    const unsigned sb = gsc_opaque(gsc_smem_u32(smraw));

    // low word of a key for the centroid in `slot`
#ifdef GSC_ONLINE_CHECKS
    unsigned long long *chk = dbg ? dbg + (long long)frames[blockIdx.x].slot * 16 + 8 : nullptr;
#endif
    auto idword = [&](int slot) -> unsigned { GSC_CHK(slot >= 0 && slot < T * CPT); return ((unsigned)gsc_lds_u16(sb + Ly::S2O + 2u * (unsigned)slot) << 16) | (unsigned)slot; };
    const GscFrame f = frames[blockIdx.x];
    const int K = f.K, N = f.N;
    if (K <= 0) return;
    if (done[f.slot]) return;                 // stopped in an earlier slice
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *cst = cnt_state + (long long)f.slot * Kmax;
    const int iter0 = passes_out[f.slot];     // passes completed by earlier slices
    const int iter_end = min(max_passes, iter0 + slice_passes);
    // cell = CPT consecutive slots of the c0-sorted codebook.  Consecutive cells go to different warps (cell c ->
    // warp c % W, lane c / W): neighbouring points have neighbouring c0, so a batch hits a few neighbouring cells
    // and this spreads them over all warps.
    const int cell = lane * (T / 32) + warp;
    const int first = cell * CPT;
    // this warp's copy of the batch thresholds / slabs
    const unsigned thrw = sb + Ly::THRW + (unsigned)warp * (GSC_ON_B * 4u);
    const unsigned xlo = sb + Ly::XLO + (unsigned)warp * (GSC_ON_B * 4u);
    const unsigned xhi = sb + Ly::XHI + (unsigned)warp * (GSC_ON_B * 4u);
    const float *Xf = X + f.chunk_off * D;
    int *lab = labels + f.chunk_off;
    float *cf = cen + (long long)f.slot * Kmax * D;

    // ---- the kernel works on a c0-SORTED copy of the codebook (c0 = first feature): slot s holds the centroid
    // with the s-th smallest c0, a thread owns a cell of CPT consecutive slots, and a point only visits the cells
    // whose c0 range meets [x0 - sqrt(U), x0 + sqrt(U)] (a centroid outside that slab has d >= (x0-c0)^2 > U).
    // Centroids drift while a pass runs; each thread keeps the exact [lo, hi] of its own c0 values, so the test
    // stays valid, only its selectivity decays -- the order is restored at the start of every pass.  Keys carry
    // the original index for the reference's tie order.
    // Start: rows in original order (slot = original index); dead slots (index >= K) are NaN and never win.
    for (int i = tid; i < KP; i += T) {
        float r[D];
#pragma unroll
        for (int k = 0; k < D; ++k) r[k] = (i < K) ? cf[(long long)i * D + k] : __int_as_float(0x7fc00000);
        gsc_sts_row<D>(sb + Ly::C + (unsigned)i * D * 4, r);
        gsc_sts_u16(sb + Ly::S2O + 2u * i, i);
        gsc_sts_i(sb + Ly::CNT + 4u * i, (iter0 > 0 && i < K) ? cst[i] : 1);  // enc:717-721 / the last pass's hits
    }
    for (int j = tid; j < N; j += T) {   // incoming guesses
        const int gg = lab[j];
        if (gg < 0 || gg >= K) lab[j] = 0;
    }
    static_assert(CPT % 2 == 0 && CPT <= 16 && DF == 4, "packed filter copy, 16-bit survivor masks");
    unsigned long long fcp[CPT / 2][DF], hp[CPT / 2];   // pairs of centroids: (2p, 2p+1)
    float c0lo = INFINITY, c0hi = -INFINITY;             // exact range of this thread's c0 values (NaN ignored)
    for (int j = tid; j < KP / 4; j += T) gsc_sts_i(sb + Ly::MFLAG + 4u * j, 0);
    gsc_sts_i(sb + Ly::DIRTY + 4u * tid, 0);
    if (tid < B) { gsc_sts_i(sb + Ly::LISTN + 4u * tid, 0); gsc_sts_u64(sb + Ly::ABEST + 8u * tid, GSC_KNONE); }
    if (tid == 0) {
        gsc_sts_d(sb + Ly::ERR, iter0 > 0 ? err_out[f.slot] : 3.40282346638528860e+38);
        gsc_sts_i(sb + Ly::STOP, 0); gsc_sts_i(sb + Ly::MODE, GSC_MODE_DONE);
    }
    __syncthreads();

    unsigned long long c_batches = 0, c_exh = 0, c_rounds = 0, c_over = 0, c_points = 0, c_cands = 0, c_again = 0;
#ifdef GSC_ONLINE_TIMING
    unsigned tm_acc[6] = {0, 0, 0, 0, 0, 0}, tm_t = 0, tm_f = 0;
#endif
    int iter = iter0;
    for (;;) {
        // The reference keeps cnts[2][K]: a pass reads cnts[not Odd(iter)] (the previous pass's hits + 1) for the
        // rates, counts into cnts[Odd(iter)] and resets the array it read to 1.  The read array is only needed for
        // the rates, which are tabulated here, so ONE array does both jobs: tabulate, reset to 1, count.
        const unsigned cnt_cur = sb + Ly::CNT;
        const double prevErr = gsc_lds_d(sb + Ly::ERR);                            // uniform copy
        // rate of every centroid for this pass (cnt_prev is constant during a pass), enc:735
        for (int j = tid; j < KP; j += T) {
            gsc_sts_f(sb + Ly::RATE + 4u * j, gsc_rate(gsc_lds_i(cnt_cur + 4u * j)));
            gsc_sts_i(cnt_cur + 4u * j, 1);
        }
        __syncthreads();
        double e_run = 0.0;   // warp 1 (thread 32's copy is used): enc:743 Double sum in point order, one batch behind the resolver
        int nbatch = 0, prev_nb = 0;

        for (int base = 0; base < N; base += GSC_ON_TP) {
            const int tn = min(GSC_ON_TP, N - base);
            __syncthreads();  // (A) previous tile fully consumed
            // ---- pass start: restore the c0 order.  Bitonic sort of (20 leading bits of c0's order key, slot) -- an
            // approximate order is all the slab test needs.  Scratch: the H region (rebuilt below) for the keys, FK for
            // the old -> new slot map.  (Re-sorting more often inside the first passes was measured: it costs more
            // than the sharper slabs save.)
            if (base == 0) {
                const unsigned sa = sb + Ly::H;
                static_assert(KP <= 4096, "12-bit slots in the sort keys");
                for (int i = tid; i < KP; i += T) {
                    const float c0 = gsc_lds_f(sb + Ly::C + (unsigned)i * D * 4);
                    gsc_sts_i(sa + 4u * i, (int)((((c0 == c0) ? gsc_fkey(c0) : 0xffffffffu) & 0xfffff000u) | (unsigned)i));
                }
                __syncthreads();
                for (int k2 = 2; k2 <= KP; k2 <<= 1)
                    for (int j = k2 >> 1; j > 0; j >>= 1) {
                        for (int i = tid; i < KP; i += T) {
                            const int l = i ^ j;
                            if (l > i) {
                                const unsigned va = (unsigned)gsc_lds_i(sa + 4u * i), vb = (unsigned)gsc_lds_i(sa + 4u * l);
                                if ((va > vb) == ((i & k2) == 0)) { gsc_sts_i(sa + 4u * i, (int)vb); gsc_sts_i(sa + 4u * l, (int)va); }
                            }
                        }
                        __syncthreads();
                    }
                // gather this thread's new cell (rows, rates, counts, original indices), scatter after everybody has read
                float rows[CPT][D], rt[CPT];
                int so[CPT], cn[CPT];
#pragma unroll
                for (int j = 0; j < CPT; ++j) {
                    const unsigned os = (unsigned)gsc_lds_i(sa + 4u * (unsigned)(first + j)) & 0xfffu;
                    gsc_lds_row<D>(sb + Ly::C + os * D * 4, rows[j]);
                    rt[j] = gsc_lds_f(sb + Ly::RATE + 4u * os);
                    cn[j] = gsc_lds_i(cnt_cur + 4u * os);
                    so[j] = gsc_lds_u16(sb + Ly::S2O + 2u * os);
                    gsc_sts_u16(sb + Ly::FK + 2u * os, first + j);   // old slot -> new slot, for the labels
                }
                __syncthreads();
                c0lo = INFINITY; c0hi = -INFINITY;
#pragma unroll
                for (int j = 0; j < CPT; ++j) {
                    const unsigned idx = (unsigned)(first + j);
                    gsc_sts_row<D>(sb + Ly::C + idx * D * 4, rows[j]);
                    gsc_sts_f(sb + Ly::RATE + 4u * idx, rt[j]);
                    gsc_sts_i(cnt_cur + 4u * idx, cn[j]);
                    gsc_sts_u16(sb + Ly::S2O + 2u * idx, so[j]);
                    if (so[j] == 0) gsc_sts_i(sb + Ly::SLOT0, (int)idx);
                    float nc = 0.0f;
#pragma unroll
                    for (int k = 0; k < DF; ++k) nc = fmaf(rows[j][k], rows[j][k], nc);
                    const float hv = -0.5f * nc * (1.0f - GSC_ON_G);
                    gsc_sts_f(sb + Ly::H + 4u * idx, hv);
                    gsc_filter_set<CPT, DF>(fcp, hp, j, rows[j], hv);
                    c0lo = fminf(c0lo, rows[j][0]); c0hi = fmaxf(c0hi, rows[j][0]);
                }
                gsc_sts_i(sb + Ly::DIRTY + 4u * cell, 0);
                for (int j = tid; j < N; j += 4 * T) {   // labels are slots (4 independent loads in flight per thread)
                    int v[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[q] = (j + q * T < N) ? lab[j + q * T] : 0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) if (j + q * T < N) lab[j + q * T] = gsc_lds_u16(sb + Ly::FK + 2u * (unsigned)v[q]);
                }
                __syncthreads();
            }
            {   // the tile's rows, 16 bytes per access, two loads in flight per thread (D is a multiple of 4: rows are 16-byte aligned)
                static_assert(D % 4 == 0, "rows copied in 16-byte pieces");
                const float4 *src = reinterpret_cast<const float4 *>(Xf + (long long)base * D);
                const int nv = tn * (D / 4);
                for (int t = tid; t < nv; t += 2 * T) {
                    const bool two = t + T < nv;
                    const float4 v0 = src[t];
                    const float4 v1 = two ? src[t + T] : make_float4(0.f, 0.f, 0.f, 0.f);
                    gsc_sts_f4(sb + Ly::X + 16u * (unsigned)t, v0);
                    if (two) gsc_sts_f4(sb + Ly::X + 16u * (unsigned)(t + T), v1);
                }
            }
            for (int t = tid; t < tn; t += T) {
                int gg = lab[base + t];
                GSC_CHK(gg >= 0 && gg < KP);
                gsc_sts_i(sb + Ly::G + 4u * t, (gg < 0 || gg >= KP) ? 0 : gg);   // slot of the previous pass's centroid
            }
            __syncthreads();  // (B)
            for (int t = tid; t < tn; t += T) {
                float nx = 0.0f;
#pragma unroll
                for (int k = 0; k < DF; ++k) { const float v = gsc_lds_f(sb + Ly::X + (unsigned)(t * D + k) * 4u); nx = fmaf(v, v, nx); }
                gsc_sts_f(sb + Ly::HX + 4u * t, 0.5f * nx * (1.0f - GSC_ON_G) - 1e-30f);
            }
            __syncthreads();  // (C)
            {   // the next tile's rows and labels (tile 0 of the next pass after the last one) start their way up the cache
                // hierarchy now: their load at the tile switch is synchronous and otherwise pays the DRAM latency
                // (measured: k-means stage -1 %; issuing it one batch before the switch instead costs a register and was no faster)
                const int nbase = (base + GSC_ON_TP < N) ? base + GSC_ON_TP : 0;
                const int nn = min(GSC_ON_TP, N - nbase);
                const char *px = reinterpret_cast<const char *>(Xf + (long long)nbase * D);
                const char *pl = reinterpret_cast<const char *>(lab + nbase);
                for (int t = tid; t < (nn * D * 4 + 127) / 128; t += T) asm volatile("prefetch.global.L1 [%0];" ::"l"(px + 128 * t));
                for (int t = tid; t < (nn * 4 + 127) / 128; t += T) asm volatile("prefetch.global.L1 [%0];" ::"l"(pl + 128 * t));
            }

            for (int pos = 0; pos < tn; pos += B) {
                const int nb = min(B, tn - pos);
#ifdef GSC_ONLINE_TIMING
                tm_f = (unsigned)clock();
#endif
                // ============ phase 0: refresh the filter copy of this thread's moved centroids ============
                {
                    const unsigned dirty = (unsigned)gsc_lds_i(sb + Ly::DIRTY + 4u * cell);
                    if (dirty) {
                        gsc_sts_i(sb + Ly::DIRTY + 4u * cell, 0);
                        // pair-wise: both centroids of a touched register pair are re-read (filter dimensions only),
                        // h_c comes from the H table the resolver keeps (same formula)
#pragma unroll
                        for (int p2 = 0; p2 < CPT / 2; ++p2)
                            if (dirty & (3u << (2 * p2))) {
                                const float4 ra = gsc_lds_f4(sb + Ly::C + (unsigned)(first + 2 * p2) * D * 4);
                                const float4 rb = gsc_lds_f4(sb + Ly::C + (unsigned)(first + 2 * p2 + 1) * D * 4);
                                fcp[p2][0] = gsc_pk2(ra.x, rb.x); fcp[p2][1] = gsc_pk2(ra.y, rb.y);
                                fcp[p2][2] = gsc_pk2(ra.z, rb.z); fcp[p2][3] = gsc_pk2(ra.w, rb.w);
                                hp[p2] = gsc_lds_u64(sb + Ly::H + (unsigned)(first + 2 * p2) * 4u);
                            }
                        c0lo = INFINITY; c0hi = -INFINITY;
#pragma unroll
                        for (int p2 = 0; p2 < CPT / 2; ++p2) {
                            float a0, a1;
                            gsc_upk2(fcp[p2][0], a0, a1);
                            c0lo = fminf(c0lo, fminf(a0, a1)); c0hi = fmaxf(c0hi, fmaxf(a0, a1));
                        }
                    }
                }
#ifdef GSC_ONLINE_CHECKS
                {   // hand-off invariants at a batch start
#pragma unroll
                    for (int p2 = 0; p2 < CPT / 2; ++p2) {
                        const float4 ra = gsc_lds_f4(sb + Ly::C + (unsigned)(first + 2 * p2) * D * 4);
                        const float4 rb = gsc_lds_f4(sb + Ly::C + (unsigned)(first + 2 * p2 + 1) * D * 4);
                        const unsigned long long want[4] = {gsc_pk2(ra.x, rb.x), gsc_pk2(ra.y, rb.y), gsc_pk2(ra.z, rb.z), gsc_pk2(ra.w, rb.w)};
#pragma unroll
                        for (int k = 0; k < 4; ++k) GSC_CHK(fcp[p2][k] == want[k]);
                        GSC_CHK(hp[p2] == gsc_lds_u64(sb + Ly::H + (unsigned)(first + 2 * p2) * 4u));
                    }
#pragma unroll
                    for (int j = 0; j < CPT; ++j) GSC_CHK(gsc_lds_u8(sb + Ly::MFLAG + (unsigned)(first + j)) == 0);
                    GSC_CHK(gsc_lds_i(sb + Ly::DIRTY + 4u * cell) == 0);
                }
#endif
                // ============ phase 1: all warps, codebook frozen ============
                float xb[D];              // lane b of every warp: point pos+b
                float Umine = INFINITY;   // ... and its bound
#pragma unroll
                for (int k = 0; k < D; ++k) xb[k] = 0.0f;
                if (lane < nb) {
                    const int p = pos + lane;
                    const int g = gsc_lds_i(sb + Ly::G + 4u * p);
                    float r[D];
                    gsc_lds_row<D>(sb + Ly::X + (unsigned)p * D * 4, xb);
                    gsc_lds_row<D>(sb + Ly::C + (unsigned)g * D * 4, r);
                    const float d = gsc_ann_dist<D>(xb, r);
                    Umine = (d == d) ? d * slack : INFINITY;   // any number is a valid threshold; see phase 2
                }
                {
                    const bool on = lane < nb && !force_exact;
                    // slab half-width: sqrt(U) widened for every rounding of the test and of the exact distance
                    const float rr = sqrtf(Umine) * 1.000002f + 4.0e-7f * fabsf(xb[0]) + 1e-30f;
                    gsc_sts_f(thrw + (unsigned)lane * 4u, on ? gsc_lds_f(sb + Ly::HX + 4u * (pos + lane)) - 0.5f * Umine : INFINITY);
                    gsc_sts_f(xlo + (unsigned)lane * 4u, on ? xb[0] - rr : INFINITY);
                    gsc_sts_f(xhi + (unsigned)lane * 4u, on ? xb[0] + rr : -INFINITY);
                }
                __syncwarp();
                // pass (a): which points' slabs meet this thread's c0 range (one bit per point, branch-free)
                unsigned hit = 0;
#pragma unroll
                for (int b4 = 0; b4 < B; b4 += 4) {
                    const float4 xl = gsc_lds_f4(xlo + (unsigned)b4 * 4u);
                    const float4 xh = gsc_lds_f4(xhi + (unsigned)b4 * 4u);
                    hit |= ((xh.x >= c0lo) && (xl.x <= c0hi)) ? (1u << b4) : 0u;
                    hit |= ((xh.y >= c0lo) && (xl.y <= c0hi)) ? (2u << b4) : 0u;
                    hit |= ((xh.z >= c0lo) && (xl.z <= c0hi)) ? (4u << b4) : 0u;
                    hit |= ((xh.w >= c0lo) && (xl.w <= c0hi)) ? (8u << b4) : 0u;
                }
                // pass (b): certified lower bounds of the cell's centroids for those points (s_c >= thr <=> lb_c <= U).
                // Survivors go to the warp's queue and are scored exactly, one per lane, at the end of the phase.
                constexpr int QCAP = (GSC_ON_B * GSC_ON_B * 8) / (4 * W);   // the FK region is free in phase 1
                const unsigned q_a = sb + Ly::FK + (unsigned)warp * (unsigned)(QCAP * 4);
                auto score_append = [&](int slot, int b) {
                    GSC_CHK(slot >= 0 && slot < KP && b >= 0 && b < nb);
                    float x[D], rw[D];
                    gsc_lds_row<D>(sb + Ly::X + (unsigned)(pos + b) * D * 4, x);
                    gsc_lds_row<D>(sb + Ly::C + (unsigned)slot * D * 4, rw);
                    const float d = gsc_ann_dist<D>(x, rw);
                    if (d == d) {
                        const unsigned long long kk = gsc_pack(__float_as_uint(d), idword(slot));
                        const int sl = gsc_atoms_add(sb + Ly::LISTN + 4u * b, 1);   // ~3 candidates per point: no contention
                        if (sl < L) {   // [slot][point]: the resolver's lanes read without bank conflicts
                            gsc_sts_u64(sb + Ly::LIST + (unsigned)(sl * B + b) * 8u, kk);
                            gsc_atoms_min_u64(sb + Ly::ABEST + 8u * (unsigned)b, kk);   // the resolver opens the batch with one load
                        }
                    }
                };
                int qn = 0;   // entries in the warp's queue (warp-uniform)
                const unsigned lt_mask = (1u << lane) - 1u;
                // all lanes call together; bits 0..15 of m are survivors of point ba, bits 16..31 of point bb
                auto push = [&](unsigned m, int fo, int ba, int bb) {
                    unsigned any;
                    while ((any = __ballot_sync(FULL, m != 0)) != 0) {
                        if (m) {
                            const int j = __ffs(m) - 1;
                            m &= m - 1;
                            const int off = qn + __popc(any & lt_mask);
                            const int slot = fo + (j & 15), b = (j < 16) ? ba : bb;
                            if (off < QCAP) gsc_sts_i(q_a + 4u * (unsigned)off, (slot << 5) | b);
                            else score_append(slot, b);
                        }
                        qn += __popc(any);
                    }
                };
                // A batch of neighbouring points hits the same few cells with most of its points; left to the owner
                // threads, one lane would work through 20+ points while its warp idles.  Cells with many points are
                // therefore evaluated by the whole warp, lane b = point b, the cell's rows broadcast from shared
                // memory; the others by their owners from the register copy, two points per trip.  The split point is
                // chosen per warp and batch from a cost model (CH per broadcast cell, CT per owner trip).
                const int cnt = __popc(hit);
                int hotT = 1;
                {
                    constexpr int CH = 300, CT = 450;
                    const int wmax = (int)__reduce_max_sync(FULL, (unsigned)cnt);
                    int bestc = 0x7fffffff;
                    const int opts[8] = {1, 3, 5, 7, 9, 13, 17, 33};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int nh = __popc(__ballot_sync(FULL, cnt >= opts[i]));
                        const int c = nh * CH + ((min(opts[i] - 1, wmax) + 1) / 2) * CT;
                        if (c < bestc) { bestc = c; hotT = opts[i]; }
                    }
                }
                const bool hot = cnt >= hotT;
                for (unsigned hm = __ballot_sync(FULL, hot); hm; hm &= hm - 1) {
                    const int o = __ffs(hm) - 1;
                    const unsigned ho = __shfl_sync(FULL, hit, o);
                    const int fo = (o * W + warp) * CPT;   // first slot of the owner's cell
                    const float thr = gsc_lds_f(thrw + (unsigned)lane * 4u);
                    unsigned m = 0;
#pragma unroll
                    for (int j4 = 0; j4 < CPT; j4 += 4) {
                        const float4 h4 = gsc_lds_f4(sb + Ly::H + (unsigned)(fo + j4) * 4u);
                        const float hh[4] = {h4.x, h4.y, h4.z, h4.w};
                        float4 c4[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) c4[j] = gsc_lds_f4(sb + Ly::C + (unsigned)(fo + j4 + j) * D * 4);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float sc = fmaf(xb[3], c4[j].w, fmaf(xb[2], c4[j].z, fmaf(xb[1], c4[j].y, fmaf(xb[0], c4[j].x, hh[j]))));
                            m |= (sc >= thr) ? (1u << (j4 + j)) : 0u;
                        }
                    }
                    if (!((ho >> lane) & 1u)) m = 0;
                    push(m, fo, lane, lane);
                }
                if (hot) hit = 0;
                __syncwarp();
                // two points per trip: their score chains are independent and hide each other's latency.  The warp makes
                // as many trips as its busiest lane needs (lanes without work carry empty masks) so that the queue
                // pushes are warp-wide.
                const int trips = (int)__reduce_max_sync(FULL, (unsigned)((__popc(hit) + 1) >> 1));
                for (int tr = 0; tr < trips; ++tr) {
                    const bool one = hit != 0;
                    const int b0 = one ? __ffs(hit) - 1 : 0;
                    hit &= hit - 1;   // (0 & -1 = 0 when there is no bit left)
                    const bool two = hit != 0;
                    const int b1 = two ? __ffs(hit) - 1 : b0;
                    hit &= hit - 1;
                    const float thr0 = gsc_lds_f(thrw + (unsigned)b0 * 4u);
                    const float thr1 = gsc_lds_f(thrw + (unsigned)b1 * 4u);
                    float s0[CPT], s1[CPT];
                    {
                        const float4 v0 = gsc_lds_f4(sb + Ly::X + (unsigned)(pos + b0) * D * 4);
                        const float4 v1 = gsc_lds_f4(sb + Ly::X + (unsigned)(pos + b1) * D * 4);
                        const float xq0[DF] = {v0.x, v0.y, v0.z, v0.w};
                        const float xq1[DF] = {v1.x, v1.y, v1.z, v1.w};
                        gsc_filter_scores<CPT, DF>(xq0, fcp, hp, s0);
                        gsc_filter_scores<CPT, DF>(xq1, fcp, hp, s1);
                    }
                    unsigned m0 = 0, m1 = 0;
#pragma unroll
                    for (int j = 0; j < CPT; ++j) { m0 |= (s0[j] >= thr0) ? (1u << j) : 0u; m1 |= (s1[j] >= thr1) ? (1u << j) : 0u; }
                    if (!one) m0 = 0;
                    if (!two) m1 = 0;
                    push(m0 | (m1 << 16), first, b0, b1);
                }
                // exact scores of the queued survivors, one per lane
                __syncwarp();
                {
                    const int qe = min(qn, QCAP);
                    for (int i = lane; i < qe; i += 32) {
                        const int e = gsc_lds_i(q_a + 4u * (unsigned)i);
                        score_append(e >> 5, e & 31);
                    }
                }
                __syncthreads();   // ---- bar 1: candidate lists complete ----
#ifdef GSC_ONLINE_TIMING
                tm_t = (unsigned)clock();
#endif
                // warp 1 adds the error terms of the previous batch while warp 0 opens this one: lane p takes point p's
                // sqrt(d / D) (the resolver only stores the distances, so the division and square root stay off its
                // path), then the terms are added in point order from registers.  Warp 1 has to be back at bar 2 before
                // warp 0 gets there; 32 dependent shared-memory loads, or 32 square roots on one thread, are not.
                if (warp == 1 && prev_nb) {
                    const unsigned eb = sb + Ly::ETB + (unsigned)(((nbatch - 1) & 1) * B) * 4u;
                    const double t = (lane < prev_nb) ? (double)sqrtf(gsc_lds_f(eb + 4u * lane) / (float)D) : 0.0;   // enc:743
#pragma unroll
                    for (int p = 0; p < B; ++p) e_run += __shfl_sync(FULL, t, p);   // (+ 0.0 past the batch's end is exact)
                }
                // ============ phase 2: the batch is resolved in rounds ============
                // warp 0 lane state: abest = best key among the list entries whose centroid has not moved
                // (or, after a re-filter, among ALL unmoved centroids: `exact`), fresh = best key among the moved
                unsigned long long abest = GSC_KNONE, fresh = GSC_KNONE, key = GSC_KNONE;
                int over = 0, exact = 0, t0 = 0, nm = 0, w = 0, pending = GSC_MODE_DONE;
                unsigned badmask = 0;
                float dkreq = INFINITY;
                float rn[D];
#pragma unroll
                for (int k = 0; k < D; ++k) rn[k] = 0.0f;
                // best key of the lane's own candidate list, skipping moved centroids (all lanes of warp 0 may call)
                int nl = 0;
                auto scan_list = [&](bool skip_moved) -> unsigned long long {
                    unsigned long long best = GSC_KNONE;
                    for (int e = 0; e < nl; e += 4) {   // 4 independent loads per trip
                        unsigned long long kq[4];
                        int mv[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) kq[q] = (e + q < nl) ? gsc_lds_u64(sb + Ly::LIST + (unsigned)((e + q) * B + lane) * 8u) : GSC_KNONE;
#pragma unroll
                        for (int q = 0; q < 4; ++q) mv[q] = (skip_moved && kq[q] != GSC_KNONE) ? gsc_lds_u8(sb + Ly::MFLAG + gsc_ks(kq[q])) : 0;
#pragma unroll
                        for (int q = 0; q < 4; ++q) if (kq[q] < best && !mv[q]) best = kq[q];
                    }
                    return best;
                };
                if (warp == 0 && lane < nb) {
                    nl = gsc_lds_i(sb + Ly::LISTN + 4u * lane);
                    abest = gsc_lds_u64(sb + Ly::ABEST + 8u * lane);   // no centroid has moved yet: the list's minimum
                    over = (nl > L) | force_exact;
                    if (tid == 0) { c_cands += nl; c_over += nl > L; }
                    nl = min(nl, L);
                    GSC_CHK(abest == scan_list(false));
                }
                const unsigned etb = sb + Ly::ETB + (unsigned)((nbatch & 1) * B) * 4u;
                for (;;) {
                    if (warp == 0) {
#ifdef GSC_ONLINE_TIMING
                        const int tm_sec = (pending == GSC_MODE_DONE) ? 0 : 3;   // first round of the batch: (a)
#endif
                        if (pending == GSC_MODE_SCAN) {
                            // ---- R3: first conflicting lane, commit the lanes before it ----
                            // Warp 0 alone issues here while the other warps wait at bar 2, and the shared-memory accessors
                            // keep source order: every load the section can issue early goes out in one trip before the
                            // commit's stores.  The committing lanes' winners are distinct (a repeated winner is a conflict),
                            // so their hit counts and moved flags are read before any of them is written.
                            const bool act = lane >= t0 && lane < nb;
                            unsigned cb = 0;
                            int cntw = 0, already = 0;
                            if (act) {
                                cb = (unsigned)gsc_lds_i(sb + Ly::CB + 4u * lane);
                                cntw = gsc_lds_i(cnt_cur + 4u * w);
                                already = gsc_lds_u8(sb + Ly::MFLAG + (unsigned)w);
                            }
                            const int tstar = min(nb, (int)__reduce_min_sync(FULL, cb ? (unsigned)(__ffs(cb) - 1) : 32u));
                            const bool commit = lane >= t0 && lane < tstar;
                            const bool takes = lane >= tstar && lane < nb;
                            if (takes) {
                                // unresolved lanes take over the fresh keys of the committed rows t0 .. tstar-1: warp ww of R2
                                // scored rows t0+ww, t0+ww+W, ... and stored running minima, so one entry per warp covers them
                                unsigned long long kq[W];
#pragma unroll
                                for (int ww = 0; ww < W; ++ww) {
                                    const int n = (tstar - t0 - ww + W - 1) / W;   // rows of warp ww below tstar (tstar > t0)
                                    kq[ww] = (n > 0) ? gsc_lds_u64(sb + Ly::FK + (unsigned)((ww * UW + n - 1) * B + lane) * 8u) : GSC_KNONE;
                                }
#pragma unroll
                                for (int ww = 0; ww < W; ++ww) if (kq[ww] < fresh) fresh = kq[ww];
                            }
                            if (commit) {
                                GSC_CHK(w >= 0 && w < KP && gsc_lds_u16(sb + Ly::S2O + 2u * (unsigned)w) < K && base + pos + lane < N);
                                gsc_sts_row<D>(sb + Ly::C + (unsigned)w * D * 4, rn);
                                {
                                    float nc = 0.0f;
#pragma unroll
                                    for (int k = 0; k < DF; ++k) nc = fmaf(rn[k], rn[k], nc);
                                    gsc_sts_f(sb + Ly::H + 4u * (unsigned)w, -0.5f * nc * (1.0f - GSC_ON_G));
                                }
                                gsc_sts_i(cnt_cur + 4u * w, cntw + 1);                // enc:744
                                lab[base + pos + lane] = w;                           // enc:742
                                gsc_sts_i(etb + 4u * lane, (int)gsc_kd(key));         // enc:743: the distance (thread 32 takes the term)
                                gsc_sts_u8(sb + Ly::MFLAG + (unsigned)w, already ? 2 : 1);   // 2: moved again in this round
                                gsc_atoms_or(sb + Ly::DIRTY + 4u * (unsigned)(w / CPT), 1u << (w % CPT));
                            }
                            const unsigned anyal = __ballot_sync(FULL, commit && already);
                            if (tid == 0) c_again += __popc(anyal);
                            {   // the moved list holds every centroid once
                                const unsigned newm = __ballot_sync(FULL, commit && !already);
                                if (commit && !already) gsc_sts_i(sb + Ly::MOVED + 4u * (unsigned)(nm + __popc(newm & ((1u << lane) - 1u))), w);
                                nm += __popc(newm);
                                GSC_CHK(nm <= B);
                            }
                            __syncwarp();
                            GSC_TM(1);
                            if (takes) {
                                // both moved flags in one trip (after the commit's stores)
                                const int mvf = (anyal && fresh != GSC_KNONE) ? gsc_lds_u8(sb + Ly::MFLAG + gsc_ks(fresh)) : 0;
                                const int mva = (abest != GSC_KNONE) ? gsc_lds_u8(sb + Ly::MFLAG + gsc_ks(abest)) : 0;
                                if (mvf == 2) {
                                    // this lane's best moved centroid moved again: its key is stale, rebuild from the moved list
                                    // (the other lanes' minima are over centroids that did not move again and stay valid)
                                    fresh = GSC_KNONE;
                                    for (int m = 0; m < nm; ++m) {
                                        const int id = gsc_lds_i(sb + Ly::MOVED + 4u * m);
                                        float rm[D];
                                        gsc_lds_row<D>(sb + Ly::C + (unsigned)id * D * 4, rm);
                                        const float d = gsc_ann_dist<D>(xb, rm);
                                        if (d == d) { const unsigned long long kk = gsc_pack(__float_as_uint(d), idword(id)); if (kk < fresh) fresh = kk; }
                                    }
                                }
                                if (mva) {
                                    // the leader among the unmoved centroids moved
                                    if (exact) { exact = 0; over = 1; abest = GSC_KNONE; }   // no list behind it: re-filter again
                                    else abest = scan_list(true);
                                }
                            }
                            if (anyal) {
                                __syncwarp();
                                if (commit && already) gsc_sts_u8(sb + Ly::MFLAG + (unsigned)w, 1);
                            }
                            t0 = tstar;
                            GSC_TM(2);
                        } else if (pending == GSC_MODE_REFILTER) {
                            // ---- R3': every re-filtered lane now knows its exact best unmoved centroid ----
                            if ((badmask >> lane) & 1u) {
                                const int i = __popc(badmask & ((1u << lane) - 1u));
                                unsigned long long k2 = GSC_KNONE;
#pragma unroll
                                for (int ww = 0; ww < W; ++ww) {
                                    const unsigned long long kk = gsc_lds_u64(sb + Ly::WKEY + (unsigned)(i * W + ww) * 8u);
                                    if (kk < k2) k2 = kk;
                                }
                                // k2 = minimum over the unmoved centroids whose lower bound is <= dkreq.  If its distance
                                // is <= dkreq (or the scan was exhaustive) it is the exact minimum over ALL unmoved
                                // centroids; otherwise all that is known is "no unmoved centroid within dkreq" (a survivor
                                // beyond dkreq says nothing about the centroids that were filtered out), and the lane is
                                // certified through Umine = dkreq like any other
                                abest = k2; over = 0;
                                exact = !(dkreq < INFINITY) || (k2 != GSC_KNONE && __uint_as_float(gsc_kd(k2)) <= dkreq);
                                if (!exact) Umine = dkreq;
                            }
                            c_exh += __popc(badmask);
                        }
                        // ---- R1: proposals of the unresolved lanes ----
                        if (t0 >= nb) {
                            // hand over to the next batch (the flags other lanes wrote above are cleared here: make the
                            // order of those stores explicit)
                            __syncwarp();
                            GSC_CHK(gsc_lds_i(sb + Ly::LISTN + 4u * lane) >= 0);
                            if (lane < nm) gsc_sts_u8(sb + Ly::MFLAG + (unsigned)gsc_lds_i(sb + Ly::MOVED + 4u * lane), 0);
                            gsc_sts_i(sb + Ly::LISTN + 4u * lane, 0);
                            gsc_sts_u64(sb + Ly::ABEST + 8u * lane, GSC_KNONE);
                            if (lane == 0) gsc_sts_i(sb + Ly::MODE, GSC_MODE_DONE);
                            pending = GSC_MODE_DONE;
                            ++c_batches; c_points += nb;
                        } else {
                            key = abest < fresh ? abest : fresh;
                            const bool okl = exact || (!over && key != GSC_KNONE && __uint_as_float(gsc_kd(key)) <= Umine);
                            if (exact && key == GSC_KNONE) key = gsc_pack(0x7f800000u, idword(gsc_lds_i(sb + Ly::SLOT0)));   // every row NaN: centroid 0, d = +inf
                            badmask = __ballot_sync(FULL, lane >= t0 && lane < nb && !okl);
                            if (badmask) {
                                // uncertified lanes: re-filter each against its best known exact distance
                                if ((badmask >> lane) & 1u) {
                                    const int i = __popc(badmask & ((1u << lane) - 1u));
                                    const float dk = (key != GSC_KNONE && !force_exact) ? __uint_as_float(gsc_kd(key)) : INFINITY;
                                    dkreq = dk;
                                    gsc_sts_i(sb + Ly::EPTS + 4u * i, pos + lane);
                                    gsc_sts_f(sb + Ly::ETHRS + 4u * i, gsc_lds_f(sb + Ly::HX + 4u * (pos + lane)) - 0.5f * dk);
                                }
                                if (lane == 0) { gsc_sts_i(sb + Ly::NE, __popc(badmask)); gsc_sts_i(sb + Ly::MODE, GSC_MODE_REFILTER); }
                                pending = GSC_MODE_REFILTER;
                            } else {
                                ++c_rounds;
                                // speculative update of every unresolved lane (enc:735-740)
                                const bool act = lane >= t0 && lane < nb;
                                w = act ? (int)gsc_ks(key) : 0;
                                gsc_lds_row<D>(sb + Ly::C + (unsigned)w * D * 4, rn);
                                const float rate = gsc_lds_f(sb + Ly::RATE + 4u * w);
#pragma unroll
                                for (int k2 = 0; k2 < D; ++k2) { float v = xb[k2] - rn[k2]; float mm = v * rate; rn[k2] = rn[k2] + mm; }
                                gsc_sts_row<D>(sb + Ly::ROWS + (unsigned)lane * D * 4, rn);
                                gsc_sts_i(sb + Ly::WS + 4u * lane, act ? (int)gsc_ki(key) : -1);   // key low word (original << 16 | slot)
                                gsc_sts_u64(sb + Ly::KEYS + 8u * lane, act ? key : GSC_KNONE);
                                if (lane == 0) { gsc_sts_i(sb + Ly::T0, t0); gsc_sts_i(sb + Ly::MODE, GSC_MODE_SCAN); }
                                pending = GSC_MODE_SCAN;
                            }
                        }
                        GSC_TM(tm_sec);
                    }
                    __syncthreads();   // ---- bar 2: proposals / request visible ----
                    const int mode = gsc_lds_i(sb + Ly::MODE);
                    if (mode == GSC_MODE_DONE) break;
                    if (mode == GSC_MODE_SCAN) {
                        // ---- R2: lane t scores the proposed rows u (warp w takes u = t0+w, t0+w+W, ...) ----
                        const int s0 = gsc_lds_i(sb + Ly::T0);
                        const unsigned long long mykey = gsc_lds_u64(sb + Ly::KEYS + 8u * lane);
                        const int myw = gsc_lds_i(sb + Ly::WS + 4u * lane);
                        int wu[UW];
                        float ru[UW][D];
#pragma unroll
                        for (int i = 0; i < UW; ++i) {
                            const int u = s0 + warp + i * W;
                            wu[i] = -2;
                            if (u < nb) { wu[i] = gsc_lds_i(sb + Ly::WS + 4u * u); gsc_lds_row<D>(sb + Ly::ROWS + (unsigned)u * D * 4, ru[i]); }
                        }
                        unsigned long long run = GSC_KNONE;
#pragma unroll
                        for (int i = 0; i < UW; ++i) {
                            const int u = s0 + warp + i * W;
                            if (u < nb) {   // uniform per warp
                                const float d = gsc_ann_dist<D>(xb, ru[i]);
                                const unsigned long long kk = (d == d) ? gsc_pack(__float_as_uint(d), (unsigned)wu[i]) : GSC_KNONE;
                                if (kk < run) run = kk;
                                gsc_sts_u64(sb + Ly::FK + (unsigned)((warp * UW + i) * B + lane) * 8u, run);
                                const bool conf = (lane > u) && (lane < nb) && ((wu[i] == myw) || (kk < mykey));
                                const unsigned cb = __ballot_sync(FULL, conf);
                                if (lane == 0) gsc_sts_i(sb + Ly::CB + 4u * u, (int)cb);
                            }
                        }
                    } else {
                        // ---- R2': re-filter the requested points with the whole CTA (threshold -inf = exhaustive) ----
                        const int ne = gsc_lds_i(sb + Ly::NE);
                        for (int i = 0; i < ne; ++i) {
                            const int pe = gsc_lds_i(sb + Ly::EPTS + 4u * i);
                            GSC_CHK(ne <= B && pe >= pos && pe < pos + nb);
                            const float thr = gsc_lds_f(sb + Ly::ETHRS + 4u * i);
                            float x[D];
                            gsc_lds_row<D>(sb + Ly::X + (unsigned)pe * D * 4, x);
                            float s[CPT];
                            {
                                const float xq[DF] = {x[0], x[1], x[2], x[3]};
                                gsc_filter_scores<CPT, DF>(xq, fcp, hp, s);
                            }
                            unsigned m = 0;
#pragma unroll
                            for (int j = 0; j < CPT; ++j) m |= (s[j] >= thr) ? (1u << j) : 0u;
                            unsigned long long best = GSC_KNONE;
                            while (m) {
                                const int j = __ffs(m) - 1;
                                m &= m - 1;
                                if (gsc_lds_u8(sb + Ly::MFLAG + (unsigned)(first + j))) continue;   // moved: covered by the fresh keys
                                float r[D];
                                gsc_lds_row<D>(sb + Ly::C + (unsigned)(first + j) * D * 4, r);
                                const float d = gsc_ann_dist<D>(x, r);
                                if (d == d) { const unsigned long long kk = gsc_pack(__float_as_uint(d), idword(first + j)); if (kk < best) best = kk; }
                            }
                            best = gsc_warp_min_key(best);
                            if (lane == 0) gsc_sts_u64(sb + Ly::WKEY + (unsigned)(i * W + warp) * 8u, best);
                        }
                    }
                    __syncthreads();   // ---- bar 3: round results complete ----
                    GSC_TM(4);
                }
#ifdef GSC_ONLINE_TIMING
                tm_acc[5] += (unsigned)clock() - tm_f;
#endif
                prev_nb = nb;
                ++nbatch;
            }
        }
        // ---- end of pass: enc:754-761 ----
        __syncthreads();
        ++iter;
#ifdef GSC_ONLINE_TIMING
        if (tid == 0 && dbg) {   // per pass: 32-bit sums do not wrap
            unsigned long long *o = dbg + (long long)f.slot * 16 + 10;
#pragma unroll
            for (int i = 0; i < 6; ++i) { o[i] += tm_acc[i]; tm_acc[i] = 0; }
        }
#endif
        if (tid == 32) {
            if (prev_nb) {
                const unsigned eb = sb + Ly::ETB + (unsigned)(((nbatch - 1) & 1) * B) * 4u;
                for (int p = 0; p < prev_nb; ++p) e_run += (double)sqrtf(gsc_lds_f(eb + 4u * p) / (float)D);   // enc:743
            }
            gsc_sts_d(sb + Ly::ERR, e_run);
            const bool same = (e_run > prevErr) ? ((e_run - prevErr) <= tol) : ((prevErr - e_run) <= tol);
            gsc_sts_i(sb + Ly::STOP, (same || iter >= max_passes) ? 1 : 0);
        }
        __syncthreads();
        if (gsc_lds_i(sb + Ly::STOP) || iter >= iter_end) break;
    }
    // the shared rows are the truth; back to the caller's order: centroid rows, hit counts and labels by original index
    for (int j = 0; j < CPT; ++j) {
        const int idx = first + j;
        const int o = gsc_lds_u16(sb + Ly::S2O + 2u * idx);
        if (o < K) {
            float r[D];
            gsc_lds_row<D>(sb + Ly::C + (unsigned)idx * D * 4, r);
#pragma unroll
            for (int k = 0; k < D; ++k) cf[(long long)o * D + k] = r[k];
            cst[o] = gsc_lds_i(sb + Ly::CNT + 4u * (unsigned)idx);
        }
    }
    for (int j = tid; j < N; j += T) {
        const int sl = lab[j];
        lab[j] = gsc_lds_u16(sb + Ly::S2O + 2u * (unsigned)((sl < 0 || sl >= KP) ? 0 : sl));
    }
    if (tid == 0) {
        passes_out[f.slot] = iter;
        err_out[f.slot] = gsc_lds_d(sb + Ly::ERR);
        done[f.slot] = gsc_lds_i(sb + Ly::STOP);
        if (dbg) {
            unsigned long long *o = dbg + (long long)f.slot * 16;
            o[0] += c_batches; o[1] += c_points; o[2] += c_exh; o[3] += c_rounds; o[4] += c_over; o[5] += c_cands; o[6] += c_again;
        }
    }
}

// ---------------------------------------------------------------------------
// Small dictionaries (K <= 256: the -cpf256 low-bitrate mode, BASELINE.json configs[2]): ONE WARP PER FRAME.
// With 256 centroids the whole codebook fits the warp's registers (lane l owns centroids l, l+32, ... l+224: 8 rows
// of D floats), so the reference's rule (enc:699-765) is run literally, one point after the other, with no
// batching, speculation or block barrier: every lane scores the point against its 8 rows in the exact operation
// order (ANN: sum (x-c)^2 left to right, two roundings per term; rows held in PAIRS as packed registers so that one
// FADD2 / FMUL2 / FFMA2-by-one serves two rows, gsc_ann_dist2), two redux steps give the nearest centroid with the lowest index on
// ties, the owning lane moves its row.  The per-batch machinery of k_online (filter, lists, resolver rounds, three
// block barriers per batch) costs more than scoring 256 centroids outright; here the warps of an SM are independent
// frames and keep its issue slots busy.  Every lane reads the point itself (one broadcast load, issued a whole point
// ahead of its use); labels are written back coalesced per tile of 32 points; the Double error sum is taken in point
// order by warp 0, one tile behind (see the pass loop).
// grid = F, block = 32 * WPF.
// ---------------------------------------------------------------------------
#define GSC_OW_CPL 8          // centroids per lane with one warp per frame (K <= 256)

// enc:735-740, 744 on one codebook row: v = x - c; m = v * rate; c = c + m (scalar: the row is one half of a packed
// pair of rows), H = 0 or 1 selects the half
template <int D, int H>
__device__ __forceinline__ void gsc_ow_update2(unsigned long long (&c2)[D], const float (&x)[D], float rate) {
#pragma unroll
    for (int k = 0; k < D; ++k) {
        float a, b;
        gsc_upk2f(c2[k], a, b);
        const float cur = H ? b : a;
        const float v = x[k] - cur;
        const float mm = v * rate;
        const float nw = cur + mm;
        c2[k] = H ? gsc_pk2f(a, nw) : gsc_pk2f(nw, b);
    }
}

// WPF warps per frame (1 or 2): with two, each warp owns half of the codebook (4 rows per lane), the two warps' best
// keys meet in shared memory (double-buffered by point parity: one 64-thread barrier per point) and the SM holds twice
// as many warps for the same number of frames -- the frame count is the only parallelism of this path.
template <int D, int WPF>
__global__ void __launch_bounds__(32 * WPF, WPF == 1 ? 10 : 8) k_online_warp(const GscFrame *__restrict__ frames, int F,
                                                                  const float *__restrict__ X,    // [sumN][D]
                                                                  float *__restrict__ cen,        // [F][Kmax][D] in/out
                                                                  int *__restrict__ labels,       // [sumN] out
                                                                  int *__restrict__ passes_out,   // [F]
                                                                  double *__restrict__ err_out,   // [F]
                                                                  double tol, int max_passes, int Kmax,
                                                                  float one) {                    // 1.0f (see gsc_ann_dist2)
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int CPL = GSC_OW_CPL / WPF;
    static_assert(CPL % 2 == 0, "rows are held in pairs");
    __shared__ unsigned long long s_key[2][2];
    __shared__ int s_stop;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned sk_mine = (unsigned)__cvta_generic_to_shared(&s_key[0][warp & 1]);
    unsigned sk_other = (unsigned)__cvta_generic_to_shared(&s_key[0][(warp & 1) ^ 1]);
    asm volatile("" : "+r"(sk_mine), "+r"(sk_other));      // computed once: not to be rematerialised (S2R) in the point loop
    const int fi = blockIdx.x;
    if (fi >= F) return;
    const GscFrame f = frames[fi];
    const int K = f.K, N = f.N;
    if (K <= 0) return;
    const float *Xf = X + f.chunk_off * D;
    int *lab = labels + f.chunk_off;
    float *cf = cen + (long long)f.slot * Kmax * D;

    // rows 2q and 2q+1 of this lane as packed pairs per coordinate (gsc_ann_dist2)
    unsigned long long c2[CPL / 2][D];
    float rate[CPL];
    int cnt[CPL];
    const unsigned long long ones = gsc_pk2f(one, one);
#pragma unroll
    for (int q = 0; q < CPL / 2; ++q) {
        const int ca = warp * (32 * CPL) + lane + 32 * (2 * q), cb = ca + 32;
#pragma unroll
        for (int k = 0; k < D; ++k)                                                                   // dead rows (NaN) never win
            c2[q][k] = gsc_pk2f((ca < K) ? cf[(long long)ca * D + k] : __int_as_float(0x7fc00000),
                                (cb < K) ? cf[(long long)cb * D + k] : __int_as_float(0x7fc00000));
        cnt[2 * q] = 1; cnt[2 * q + 1] = 1;                                                           // enc:717-721
    }
    double err = 3.40282346638528860e+38;   // enc:724 (warp 0 carries it)
    int iter = 0;
    for (;;) {
        const double prevErr = err;
#pragma unroll
        for (int j = 0; j < CPL; ++j) { rate[j] = gsc_rate(cnt[j]); cnt[j] = 1; }   // enc:735 (cnt_prev is constant during a pass), 754-758
        // enc:743 err += sqrt(d / D), in point order, Double.  The square roots of a tile of 32 points are taken by the
        // 32 lanes at once after the tile (lane l keeps point l's distance), and the ordered Double additions of that
        // tile ride along with the next tile's points, one per point: 3 instructions per point in warp 0 instead of a
        // sqrt + convert + add in every thread, and off the dependency chain of the centroids.
        double e_run = 0.0, es_prev = 0.0;
        int tn_prev = 0;
        int par = 0;
        float xn[D];
#pragma unroll
        for (int k = 0; k < D; ++k) xn[k] = 0.0f;
        if (N > 0) gsc_load_row<D>(Xf, 0, xn);                                              // every lane the same row: one broadcast load
        for (int base = 0; base < N; base += 32) {
            const int tn = min(32, N - base);
            int mylab = 0;
            float mydw = 0.0f;
#pragma unroll 2
            for (int p = 0; p < tn; ++p, par ^= 1) {
                float x[D];
#pragma unroll
                for (int k = 0; k < D; ++k) x[k] = xn[k];
                gsc_load_row<D>(Xf, min(base + p + 1, N - 1), xn);                  // the next point, a whole step ahead of its use
                // nearest of this lane's rows: ascending j = ascending centroid index, strict < keeps the lowest
                // (two half-length compare chains merged with a strict <: the same winner as one chain, half the depth)
                float bd = INFINITY, bdh = INFINITY;
                int bj = -1, bjh = -1;
                {
                    // gsc_ann_dist2 for all row pairs, written dimension by dimension so that the CPL/2 independent
                    // chains advance together (one pair after the other leaves dependent packed ops back to back)
                    unsigned long long d2[CPL / 2];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        unsigned long long t[CPL / 2], mq[CPL / 2];
                        const unsigned long long xk = gsc_pk2f(x[k], x[k]);
#pragma unroll
                        for (int q = 0; q < CPL / 2; ++q) asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(t[q]) : "l"(xk), "l"(c2[q][k]));
#pragma unroll
                        for (int q = 0; q < CPL / 2; ++q) asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(mq[q]) : "l"(t[q]), "l"(t[q]));
#pragma unroll
                        for (int q = 0; q < CPL / 2; ++q) {
                            if (k == 0) d2[q] = mq[q];          // 0 + m == m: a square is +0, positive or NaN
                            else asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d2[q]) : "l"(mq[q]), "l"(ones), "l"(d2[q]));
                        }
                    }
#pragma unroll
                    for (int q = 0; q < CPL / 2; ++q) {
                        float da, db;
                        gsc_upk2f(d2[q], da, db);
                        if (CPL < 8 || q < CPL / 4) {
                            if (da < bd) { bd = da; bj = 2 * q; }
                            if (db < bd) { bd = db; bj = 2 * q + 1; }
                        } else {
                            if (da < bdh) { bdh = da; bjh = 2 * q; }
                            if (db < bdh) { bdh = db; bjh = 2 * q + 1; }
                        }
                    }
                }
                if (bdh < bd) { bd = bdh; bj = bjh; }
                const unsigned dk = (bj >= 0) ? __float_as_uint(bd) : 0xffffffffu;      // distances are >= 0: bits order them
                unsigned m = __reduce_min_sync(FULL, dk);
                unsigned ci = __reduce_min_sync(FULL, (dk == m && bj >= 0) ? (unsigned)(warp * (32 * CPL) + lane + 32 * bj) : 0xffffffffu);
                if (WPF == 2) {
                    // the two warps' (distance, index) keys meet in shared memory: slot [par][warp], 8 bytes each
                    if (lane == 0) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(sk_mine + 16u * par), "r"(ci), "r"(m) : "memory");
                    __syncthreads();
                    unsigned oc, om;
                    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(oc), "=r"(om) : "r"(sk_other + 16u * par) : "memory");
                    const bool take = (om < m) || (om == m && oc < ci);
                    m = take ? om : m; ci = take ? oc : ci;
                }
                float dw = __uint_as_float(m);
                if (ci == 0xffffffffu) { ci = 0; dw = INFINITY; }                        // every row NaN: centroid 0, d = +inf
                const int win = (int)ci;
                constexpr int LOG_CPL = (CPL == 8) ? 3 : (CPL == 4) ? 2 : (CPL == 2) ? 1 : 0;
                static_assert((1 << LOG_CPL) == CPL, "rows per lane must be a power of two");
                if ((unsigned)warp == (ci >> (5 + LOG_CPL)) && (unsigned)lane == (ci & 31u)) {
                    // enc:735-740, 744 on the winning row (static register indices: a branch tree over the owned rows)
                    const unsigned wj = (ci >> 5) & (unsigned)(CPL - 1);
#define GSC_OW_UPD(J) { gsc_ow_update2<D, ((J) < CPL ? (J) : 0) & 1>(c2[((J) < CPL ? (J) : 0) >> 1], x, rate[(J) < CPL ? (J) : 0]); cnt[(J) < CPL ? (J) : 0] += 1; }
                    if (CPL <= 4 || wj < 4) {
                        if (CPL <= 2 || (wj & 3u) < 2) { if (CPL <= 1 || (wj & 1u) == 0) GSC_OW_UPD(0) else GSC_OW_UPD(1) }
                        else { if ((wj & 1u) == 0) GSC_OW_UPD(2) else GSC_OW_UPD(3) }
                    } else {
                        if ((wj & 3u) < 2) { if ((wj & 1u) == 0) GSC_OW_UPD(4) else GSC_OW_UPD(5) }
                        else { if ((wj & 1u) == 0) GSC_OW_UPD(6) else GSC_OW_UPD(7) }
                    }
#undef GSC_OW_UPD
                }
                if (lane == p) { mylab = win; mydw = dw; }                              // enc:742
                const double ev = __shfl_sync(FULL, es_prev, p);
                if (p < tn_prev) e_run += ev;                                           // only warp 0's sum is used
            }
            if (warp == 0) {
                for (int p = tn; p < tn_prev; ++p) e_run += __shfl_sync(FULL, es_prev, p);   // only when the last tile is short
                if (lane < tn) lab[base + lane] = mylab;
                es_prev = (double)sqrtf(mydw / (float)D);
                tn_prev = tn;
            }
        }
        bool same = false;
        if (warp == 0) {
            for (int p = 0; p < tn_prev; ++p) e_run += __shfl_sync(FULL, es_prev, p);
            err = e_run;
            same = (err > prevErr) ? ((err - prevErr) <= tol) : ((prevErr - err) <= tol);   // enc:761
        }
        ++iter;
        if (WPF == 2) {
            if (threadIdx.x == 0) s_stop = same ? 1 : 0;
            __syncthreads();
            same = s_stop != 0;
        }
        if (same || iter >= max_passes) break;
    }
#pragma unroll
    for (int q = 0; q < CPL / 2; ++q) {
        const int ca = warp * (32 * CPL) + lane + 32 * (2 * q), cb = ca + 32;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            float a, b;
            gsc_upk2f(c2[q][k], a, b);
            if (ca < K) cf[(long long)ca * D + k] = a;
            if (cb < K) cf[(long long)cb * D + k] = b;
        }
    }
    if (threadIdx.x == 0) { passes_out[f.slot] = iter; err_out[f.slot] = err; }
}
