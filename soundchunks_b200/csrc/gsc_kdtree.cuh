// gsc_kdtree.cuh -- kmeans_mode 3: the ANN 1.1.2 kd-tree searches of the reference binary on the device, bit for bit
// with the CPU oracle's restatement of ANN's kd_tree.cpp / kd_split.cpp / kd_util.cpp / kd_search.cpp (its ann_build,
// ann_search_rec, ann_ksearch_rec and the kd-tree forms of KNNScanReduce and KNNFit).
//
// Tree layout.  Bucket size 1 and n_lo = n / 2 make the shape a function of n alone, so children are implicit: the
// internal node over the range [off, off + n) (n >= 2) is numbered by its split gap off + n/2 - 1 (n - 1 internal
// nodes, numbers 0 .. n-2) and stores its cut dimension, cut value and the two bounds of its own box in that
// dimension; a range of one position is the leaf pidx[off].  pidx is the point order the median splits leave behind.
// The same code builds the KNNScanReduce tree over the centroids (shared memory) and the KNNFit tree over the 4R
// variant rows (global memory).
#pragma once
#include "gsc_device.cuh"
#include "gsc_kernels.cuh"   // gsc_knnfit_epsilon, gsc_in_band
#include "gsc_online.cuh"    // gsc_rate

#define GSC_KDT_THREADS 128   // k_kdt_scan CTA: every thread builds, warp 0 searches
#define GSC_KDT_STK 16        // DFS stack entries per search: trees of up to 65,536 points
#define GSC_KDT_VCAP 64       // leaves a speculative lane records (a longer visit is uncertified, unless it is lane 0)
#define GSC_KDT_MAXF 3.40282346638528860e+38f

template <int D>
__device__ __forceinline__ float gsc_kdt_sel(const float (&v)[D], int c) {
    float r = v[0];
#pragma unroll
    for (int d = 1; d < D; ++d) if (d == c) r = v[d];
    return r;
}

// ann_build over pts[n][D] by all threads of the CTA (n <= 65,536): annEnclRect (one thread per dimension, the scan
// as written), then the nodes depth by depth, each node by one thread running kd_split / annMaxSpread /
// annMedianSplit exactly as the sequential code (the quickselect's swap sequence decides which of equal values land
// left or right, hence the leaf order and the visit order that breaks ties).  A node's box is the enclosing
// rectangle with its ancestors' cuts applied from the root down, which is what the recursion's bb_lo / bb_hi hold.
// bb[2D]: lo | hi of the enclosing rectangle.  Ends with a CTA barrier.
template <int D>
__device__ void gsc_kdt_build(const float *pts, int n, unsigned short *pidx, unsigned char *cd, float *cv, float *lob,
                              float *hib, float *bb) {
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < n; i += nt) pidx[i] = (unsigned short)i;
    if (tid < D) {
        float lo = pts[tid], hi = lo;
        for (int i = 0; i < n; ++i) {
            const float c = pts[(long long)i * D + tid];
            if (c < lo) lo = c; else if (c > hi) hi = c;
        }
        bb[tid] = lo; bb[D + tid] = hi;
    }
    __syncthreads();
    for (int lev = 0; (1 << lev) < n; ++lev) {
        for (int j = tid; j < (1 << lev); j += nt) {
            float lo[D], hi[D];
#pragma unroll
            for (int d = 0; d < D; ++d) { lo[d] = bb[d]; hi[d] = bb[D + d]; }
            int off = 0, m = n;
            for (int b = lev - 1; b >= 0 && m >= 2; --b) {       // root -> node j of this depth
                const int h = m / 2, g = off + h - 1, c = cd[g];
                const float v = cv[g];
                if ((j >> b) & 1) {
#pragma unroll
                    for (int d = 0; d < D; ++d) if (d == c) lo[d] = v;
                    off += h; m -= h;
                } else {
#pragma unroll
                    for (int d = 0; d < D; ++d) if (d == c) hi[d] = v;
                    m = h;
                }
            }
            if (m < 2) continue;                                  // a leaf above this depth, or this depth's leaf
            unsigned short *px = pidx + off;
            // annMaxSpread
            int cdim = 0;
            float max_spr = 0.0f;
#pragma unroll 1
            for (int d = 0; d < D; ++d) {
                float mn = pts[(int)px[0] * D + d], mx = mn;
                for (int i = 1; i < m; ++i) {
                    const float c = pts[(int)px[i] * D + d];
                    if (c < mn) mn = c; else if (c > mx) mx = c;
                }
                const float spr = mx - mn;
                if (spr > max_spr) { max_spr = spr; cdim = d; }
            }
            // annMedianSplit (with the oracle's two bounds for NaN rows)
            const float *pc = pts + cdim;
            const int n_lo = m / 2;
#define PAV(i) pc[(int)px[(i)] * D]
#define PASWAP(a, b) do { const unsigned short t_ = px[(a)]; px[(a)] = px[(b)]; px[(b)] = t_; } while (0)
            int l = 0, r = m - 1;
            while (l < r) {
                int i = (r + l) / 2, k;
                if (PAV(i) > PAV(r)) PASWAP(i, r);
                PASWAP(l, i);
                const float c = PAV(l);
                i = l; k = r;
                for (;;) {
                    while (i < r && PAV(++i) < c) ;
                    while (k > l && PAV(--k) > c) ;
                    if (i < k) PASWAP(i, k); else break;
                }
                PASWAP(l, k);
                if (k > n_lo) r = k - 1;
                else if (k < n_lo) l = k + 1;
                else break;
            }
            {
                float c = PAV(0);
                int k = 0;
                for (int i = 1; i < n_lo; ++i) if (PAV(i) > c) { c = PAV(i); k = i; }
                PASWAP(n_lo - 1, k);
            }
            const float cut = (float)(((double)PAV(n_lo - 1) + (double)PAV(n_lo)) / 2.0);
#undef PAV
#undef PASWAP
            const int g = off + n_lo - 1;
            cd[g] = (unsigned char)cdim; cv[g] = cut; lob[g] = gsc_kdt_sel<D>(lo, cdim); hib[g] = gsc_kdt_sel<D>(hi, cdim);
        }
        __syncthreads();
    }
}

// annBoxDistance of q from the enclosing rectangle
template <int D>
__device__ __forceinline__ float gsc_kdt_box_dist(const float (&q)[D], const float *bb) {
    float bd = 0.0f;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        if (q[d] < bb[d]) { const float tt = bb[d] - q[d]; bd = bd + tt * tt; }
        else if (q[d] > bb[D + d]) { const float tt = q[d] - bb[D + d]; bd = bd + tt * tt; }
    }
    return bd;
}

// One step down from the internal node (off, m): the near child becomes (off, m), the far child and its box distance
// go on the stack.  The recursion computes that distance after the near subtree returns, but it depends on nothing
// the subtree changes, so the check against the (then current) bound happens at the pop.
template <int D>
__device__ __forceinline__ void gsc_kdt_descend(const float (&q)[D], const unsigned char *cd, const float *cv,
                                                const float *lob, const float *hib, int &off, int &m, float bd,
                                                unsigned *stk, float *stkd, int &sp) {
    const int h = m / 2, g = off + h - 1;
    const float qc = gsc_kdt_sel<D>(q, cd[g]);
    const float cut_diff = qc - cv[g];
    float box_diff;
    unsigned far;
    if (cut_diff < 0) {
        box_diff = lob[g] - qc;
        far = ((unsigned)(off + h) << 16) | (unsigned)(m - h);
        m = h;
    } else {
        box_diff = qc - hib[g];
        far = ((unsigned)off << 16) | (unsigned)h;
        off += h; m -= h;
    }
    if (box_diff < 0) box_diff = 0;
    stk[sp] = far;
    stkd[sp] = bd + (cut_diff * cut_diff - box_diff * box_diff);
    ++sp;
}

// ann_search1: nearest point, ties to the first point visited.  Leaves read the rows as they are now.  The first
// GSC_KDT_VCAP visited points go to vis[]; nvis counts them all.  Returns -1 only where the oracle does.
template <int D>
__device__ __forceinline__ int gsc_kdt_search1(const float (&q)[D], const float *rows, int n, const unsigned short *pidx,
                                               const unsigned char *cd, const float *cv, const float *lob,
                                               const float *hib, const float *bb, unsigned *stk, float *stkd,
                                               unsigned short *vis, int &nvis, float &best) {
    float bd = gsc_kdt_box_dist<D>(q, bb);
    best = GSC_KDT_MAXF;
    int idx = -1, off = 0, m = n, sp = 0;
    nvis = 0;
    for (;;) {
        while (m >= 2) gsc_kdt_descend<D>(q, cd, cv, lob, hib, off, m, bd, stk, stkd, sp);
        const int p = pidx[off];                                  // ANNkd_leaf::ann_search
        if (nvis < GSC_KDT_VCAP) vis[nvis] = (unsigned short)p;
        ++nvis;
        const float *pp = rows + p * D;
        const float min_dist = best;
        float dist = 0.0f;
        bool full = true;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            if (full) {
                const float tt = q[d] - pp[d];
                const float mm = tt * tt;
                dist = dist + mm;
                if (dist > min_dist) full = false;
            }
        }
        if (full && idx < 0) { best = dist; idx = p; }
        else if (full && dist < best) { best = dist; idx = p; }
        bool more = false;
        while (sp > 0) {
            --sp;
            if (stkd[sp] < best) { off = (int)(stk[sp] >> 16); m = (int)(stk[sp] & 0xffffu); bd = stkd[sp]; more = true; break; }
        }
        if (!more) break;
    }
    return idx;
}

// ---------------------------------------------------------------------------
// KNNScanReduce (enc:699-765) through the tree, one CTA per frame.
//
// Speculation.  A query reads nothing but the tree (fixed for the pass) and the rows of the leaves it visits; if none
// of those rows changed, its whole trajectory -- every comparison, the answer, the distance -- is the same.  So warp 0
// searches up to 32 consecutive points at once against the rows as they stand, each lane recording its visited
// leaves.  Lane t is certified iff no earlier lane of the round chose a centroid that lane t visited or chose itself
// (and its list did not overflow; lane 0 is always right).  The lanes before the first uncertified one commit in
// point order -- row updates, labels, counts, err -- and their centroids are distinct; the rest are searched again
// in the next round.  lanes = 1 (GSC_DBG_KDTREE_SERIAL) is the plain sequential rule.
// ---------------------------------------------------------------------------
struct GscKdtScanSmem {
    unsigned rows, rate, cv, lob, hib, stk, stkd, pidx, vis, cd, own, total;
    __host__ __device__ GscKdtScanSmem(int K, int D) {
        unsigned o = 0;
        rows = o; o += 4u * K * D;
        rate = o; o += 4u * K;
        cv = o; o += 4u * K;
        lob = o; o += 4u * K;
        hib = o; o += 4u * K;
        stk = o; o += 4u * 32 * GSC_KDT_STK;
        stkd = o; o += 4u * 32 * GSC_KDT_STK;
        pidx = o; o += 2u * K;
        vis = o; o += 2u * 32 * GSC_KDT_VCAP;
        cd = o; o += K;
        own = o; o += K;
        total = (o + 15u) & ~15u;
    }
};

template <int D>
__global__ void __launch_bounds__(GSC_KDT_THREADS, 1) k_kdt_scan(const GscFrame *__restrict__ frames,
                                                              const float *__restrict__ X,    // [sumN][D]
                                                              float *__restrict__ cen,        // [F][Kmax][D] in/out
                                                              int *__restrict__ labels,       // [sumN] out
                                                              int *__restrict__ passes_out,   // [F]
                                                              double *__restrict__ err_out,   // [F]
                                                              int *__restrict__ cnt,          // [F][Kmax] scratch
                                                              double tol, int max_passes, int Kmax, int lanes,
                                                              unsigned long long *__restrict__ dbg) {  // [F][16]
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ float s_bb[2 * D];
    __shared__ int s_stop;
    const GscFrame f = frames[blockIdx.x];
    const int K = f.K, N = f.N;
    if (K <= 0) return;                                           // passthrough frame (passes / err zeroed by the caller)
    const GscKdtScanSmem Ly(Kmax, D);
    float *rows = reinterpret_cast<float *>(s_raw + Ly.rows), *rate = reinterpret_cast<float *>(s_raw + Ly.rate);
    float *cv = reinterpret_cast<float *>(s_raw + Ly.cv), *lob = reinterpret_cast<float *>(s_raw + Ly.lob);
    float *hib = reinterpret_cast<float *>(s_raw + Ly.hib);
    unsigned short *pidx = reinterpret_cast<unsigned short *>(s_raw + Ly.pidx);
    unsigned char *cd = s_raw + Ly.cd, *own = s_raw + Ly.own;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned *stk = reinterpret_cast<unsigned *>(s_raw + Ly.stk) + lane * GSC_KDT_STK;
    float *stkd = reinterpret_cast<float *>(s_raw + Ly.stkd) + lane * GSC_KDT_STK;
    unsigned short *vis = reinterpret_cast<unsigned short *>(s_raw + Ly.vis) + lane * GSC_KDT_VCAP;
    float *cf = cen + (long long)f.slot * Kmax * D;
    int *cntf = cnt + (long long)f.slot * Kmax;
    const float *Xf = X + f.chunk_off * D;
    int *lab = labels + f.chunk_off;
    for (int t = threadIdx.x; t < K * D; t += blockDim.x) rows[t] = cf[t];
    for (int t = threadIdx.x; t < K; t += blockDim.x) { cntf[t] = 1; own[t] = 0xff; }   // enc:717-721
    double err = 3.40282346638528860e+38;                        // enc:724 (thread 0 carries it)
    int iter = 0;
    unsigned long long n_rounds = 0, n_points = 0, n_search = 0, n_over = 0;
    for (;;) {
        const double prevErr = err;
        __syncthreads();
        // enc:735: the rate of a centroid is fixed for the pass (last pass's count); the counts restart at 1 (enc:754-758)
        for (int t = threadIdx.x; t < K; t += blockDim.x) { rate[t] = gsc_rate(cntf[t]); cntf[t] = 1; }
        gsc_kdt_build<D>(rows, K, pidx, cd, cv, lob, hib, s_bb); // enc:729, from the rows at the start of the pass
        if (warp == 0) {
            double e_run = 0.0;
            for (int base = 0; base < N;) {
                const int i = base + lane;
                const bool act = lane < lanes && i < N;
                int bi = -1, nv = 0;
                float best = 0.0f, x[D];
#pragma unroll
                for (int k = 0; k < D; ++k) x[k] = 0.0f;
                if (act) {
#pragma unroll
                    for (int k = 0; k < D; ++k) x[k] = Xf[(long long)i * D + k];
                    bi = gsc_kdt_search1<D>(x, rows, K, pidx, cd, cv, lob, hib, s_bb, stk, stkd, vis, nv, best);   // enc:733
                    if (bi < 0) { bi = 0; best = 0.0f; }
                }
                const unsigned am = __ballot_sync(FULL, act);
                // own[c] = the lowest lane of the round that chose c
                const unsigned grp = __match_any_sync(FULL, act ? bi : -1 - lane);
                const bool leader = act && lane == __ffs(grp) - 1;
                if (leader) own[bi] = (unsigned char)lane;
                __syncwarp();
                bool ok = act;
                if (act && lane > 0) {
                    ok = nv <= GSC_KDT_VCAP && own[bi] >= lane;
                    for (int v = 0; ok && v < nv; ++v) ok = own[vis[v]] >= lane;
                }
                const unsigned bad = __ballot_sync(FULL, act && !ok);
                const int nc = bad ? __ffs(bad) - 1 : __popc(am);
                n_over += __popc(__ballot_sync(FULL, act && nv > GSC_KDT_VCAP));
                __syncwarp();
                if (leader) own[bi] = 0xff;
                double ev = 0.0;
                if (lane < nc) {
                    const float r = rate[bi];
                    float *c = rows + bi * D;
#pragma unroll
                    for (int k = 0; k < D; ++k) { const float v = x[k] - c[k]; const float mm = v * r; c[k] = c[k] + mm; }   // enc:736-740
                    lab[i] = bi;                                                                                     // enc:742
                    cntf[bi] += 1;                                                                                   // enc:744
                    ev = (double)sqrtf(best / (float)D);
                }
                for (int p = 0; p < nc; ++p) e_run += __shfl_sync(FULL, ev, p);                                     // enc:743, point order
                base += nc;
                ++n_rounds; n_points += (unsigned long long)nc; n_search += (unsigned long long)__popc(am);
                __syncwarp();
            }
            if (threadIdx.x == 0) {
                err = e_run;
                const bool same = (err > prevErr) ? ((err - prevErr) <= tol) : ((prevErr - err) <= tol);   // enc:761
                s_stop = (same || iter + 1 >= max_passes) ? 1 : 0;
            }
        }
        ++iter;
        __syncthreads();
        if (s_stop) break;
    }
    for (int t = threadIdx.x; t < K * D; t += blockDim.x) cf[t] = rows[t];
    if (threadIdx.x == 0) {
        passes_out[f.slot] = iter;
        err_out[f.slot] = err;
        if (dbg) {
            unsigned long long *o = dbg + (long long)f.slot * 16;
            o[0] = n_rounds; o[1] = n_points; o[2] = n_search; o[3] = n_over;
        }
    }
}

// ---------------------------------------------------------------------------
// KNNFit (enc:915-965) through the tree: one tree per frame over the 4R variant rows
// (row = entry*4 + neg*2 + rev), in global memory; one thread per query.
// Storage per frame, Mmax = 4*Kmax rows: V [Mmax][CS] | nodes cv, lob, hib [3][Mmax] | pidx [Mmax] | cd [Mmax] |
// bb [2*CS].
// ---------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(256, 1) k_kdt_fit_build(const GscFrame *__restrict__ frames, int bits,
                                                       const int *__restrict__ divider,
                                                       const short *__restrict__ dict,
                                                       const unsigned char *__restrict__ datten,
                                                       float *__restrict__ V, float *__restrict__ nodes,
                                                       unsigned short *__restrict__ pidx, unsigned char *__restrict__ cd,
                                                       float *__restrict__ bb, int Kmax) {
    const GscFrame f = frames[blockIdx.x];
    const long long fo = (long long)f.slot * Kmax, Mmax = 4LL * Kmax;
    const int R = f.R, M = 4 * R;
    float *Vf = V + f.slot * Mmax * CS, *nf = nodes + f.slot * 3 * Mmax;
    GscLaw L;
    L.init(1.0 / (double)divider[f.slot]);
    const int obd = (1 << (bits - 1)) - 1;
    for (int t = threadIdx.x; t < 2 * R * CS; t += blockDim.x) {   // the variant rows (enc:930-938)
        const int i = t / CS, j = t - i * CS, e = i >> 1;
        const bool ng = (i & 1) != 0;
        const double coeff = L.T[datten[fo + e]];
        Vf[((long long)i * 2 + 0) * CS + j] = (float)gsc_dequant(dict[(fo + e) * CS + j], obd, coeff, ng);
        Vf[((long long)i * 2 + 1) * CS + j] = (float)gsc_dequant(dict[(fo + e) * CS + CS - 1 - j], obd, coeff, ng);
    }
    __syncthreads();
    gsc_kdt_build<CS>(Vf, M, pidx + f.slot * Mmax, cd + f.slot * Mmax, nf, nf + Mmax, nf + 2 * Mmax, bb + f.slot * 2 * CS);
}

template <int CS>
__global__ void __launch_bounds__(128) k_kdt_fit(const GscFrame *__restrict__ frames, const short *__restrict__ pcm,
                                                 int bits, const int *__restrict__ divider,
                                                 const float *__restrict__ V, const float *__restrict__ nodes,
                                                 const unsigned short *__restrict__ pidx,
                                                 const unsigned char *__restrict__ cd, const float *__restrict__ bb,
                                                 int *__restrict__ best,   // [sumN]
                                                 int *__restrict__ use,    // [F][Kmax], zeroed
                                                 int Kmax) {
    const GscFrame f = frames[blockIdx.y];
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= f.N) return;
    const long long fo = (long long)f.slot * Kmax, Mmax = 4LL * Kmax;
    const int M = 4 * f.R;
    const float *Vf = V + f.slot * Mmax * CS, *nf = nodes + f.slot * 3 * Mmax, *bbf = bb + f.slot * 2 * CS;
    const float *cv = nf, *lob = nf + Mmax, *hib = nf + 2 * Mmax;
    const unsigned short *px = pidx + f.slot * Mmax;
    const unsigned char *cdf = cd + f.slot * Mmax;
    const int i = n / f.C, ch = n - i * f.C;
    const short *row = pcm + f.pcm_off + (long long)ch * f.stride + (long long)i * CS;
    float q[CS];
#pragma unroll
    for (int j = 0; j < CS; ++j) q[j] = (i * CS + j < f.S) ? (float)gsc_sample(row[j]) : 0.0f;   // enc:949-950
    // ann_ksearch_rec, k = min(64, M): ANNmin_k insertion list, equal keys in visit order
    const int kk = M < GSC_BUCKET ? M : GSC_BUCKET;
    float key[GSC_BUCKET];
    int kid[GSC_BUCKET];
    unsigned stk[GSC_KDT_STK];
    float stkd[GSC_KDT_STK];
    int kn = 0, off = 0, m = M, sp = 0;
    float bd = gsc_kdt_box_dist<CS>(q, bbf);
    for (;;) {
        while (m >= 2) gsc_kdt_descend<CS>(q, cdf, cv, lob, hib, off, m, bd, stk, stkd, sp);
        const int p = px[off];
        const float *pp = Vf + (long long)p * CS;
        const float min_dist = (kn == kk) ? key[kk - 1] : GSC_KDT_MAXF;
        float dist = 0.0f;
        bool full = true;
#pragma unroll
        for (int d = 0; d < CS; ++d) {
            if (full) {
                const float tt = q[d] - pp[d];
                const float mm = tt * tt;
                dist = dist + mm;
                if (dist > min_dist) full = false;
            }
        }
        if (full) {                                               // ANNmin_k::insert
            int s;
            for (s = kn; s > 0; --s) {
                if (key[s - 1] > dist) { if (s < kk) { key[s] = key[s - 1]; kid[s] = kid[s - 1]; } }
                else break;
            }
            if (s < kk) { key[s] = dist; kid[s] = p; }
            if (kn < kk) ++kn;
        }
        bool more = false;
        while (sp > 0) {
            --sp;
            const float kth = (kn == kk) ? key[kk - 1] : GSC_KDT_MAXF;
            if (stkd[sp] < kth) { off = (int)(stk[sp] >> 16); m = (int)(stk[sp] & 0xffffu); bd = stkd[sp]; more = true; break; }
        }
        if (!more) break;
    }
    // enc:954-958: lowest row index among the candidates within epsilon of the nearest
    const float eps = gsc_knnfit_epsilon(bits, 1.0 / (double)divider[f.slot]);
    const float fcs = (float)CS;
    int b = 0;
    if (kn > 0) {
        const float a = sqrtf(key[0] / fcs);
        b = kid[0];
        for (int j = 1; j < kn; ++j)
            if (gsc_in_band(a, key[j], fcs, eps) && kid[j] < b) b = kid[j];
    }
    best[f.chunk_off + n] = b;
    atomicAdd(&use[fo + (b >> 2)], 1);                            // enc:962-964
}
