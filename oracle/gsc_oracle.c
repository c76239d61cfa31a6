/*
 * gsc_oracle.c -- CPU restatement of the SoundChunks encoder hot path.
 *
 * TEST INFRASTRUCTURE ONLY (see gsc_oracle.h).  PARITY UNPINNED: there are no
 * reference golden vectors for this path and the reference cannot run here.
 * Third-party algorithms restated from their published sources because the
 * reference ships them as binaries only: yakmo (N. Yoshinaga; GliGli's DLL fork,
 * yakmo_single.dll, no version pin) and ANN 1.1.2 (D. Mount, S. Arya; ANN.dll).
 *
 * Citations:  enc:L = /root/reference/encoder/encoder.lpr line L
 *             dec:L = /root/reference/decoder/decoder.lpr line L
 * Build with -ffp-contract=off: the reference is FreePascal/MSVC x86-64 SSE2
 * scalar code without fused multiply-add.
 *
 * FreePascal typing rules that matter here (x86-64, SSE):
 *   round()            half-to-even               -> nearbyint()
 *   Single op Integer  evaluated in Single
 *   sqrt(Single)       Single;  sqrt(Integer) Double
 *   IsZero(Double)     |x| <= 1e-12
 *   SameValue(a,b,e)   |a-b| <= e  (in the operands' type)
 *   math.log10(x)      ln(x) * 0.43429448190325182765
 */
#include "gsc_oracle.h"
/* the one routine shared with the product: a correctly-rounded ln in plain IEEE double operations, so that the
 * cepstral features do not depend on whose libm evaluated log() (checked against mpmath, tests/test_log_cr.py) */
#include "../soundchunks_b200/csrc/gsc_log.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define GSC_MAX_ATTENUATION 15      /* enc:14 */
#define GSC_MAX_CHUNKS 4096         /* enc:15 */
#define GSC_BUCKET 64               /* enc:917 CBucketSize */
#define GSC_PI 3.14159265358979323846

/* ------------------------------------------------------------------ */
/* scalar sample functions                                            */
/* ------------------------------------------------------------------ */

double gsc_ref_log_cr(double x) { return gsc_log_cr(x); }

/* enc:1643-1646 */
double gsc_ref_float_sample(int16_t s) { return (double)s / 32767.0; }

/* enc:1638-1641 */
int16_t gsc_ref_make16(double smp)
{
    double r = nearbyint(smp * 32767.0);
    if (r < -32768.0) r = -32768.0;
    if (r > 32767.0) r = 32767.0;
    return (int16_t)r;
}

/* enc:1654-1656 / 1671-1673: coeff := 1.0; for i := 0 to a do coeff += i*Law */
static double atten_coeff(int a, double law)
{
    double c = 1.0;
    for (int i = 0; i <= a; ++i) c += (double)i * law;
    return c;
}

/* enc:1648-1663 makeOutputSample */
int16_t gsc_ref_quant(double smp, int bits, int atten, int neg, double law)
{
    double coeff = atten_coeff(atten, law);
    int obd = (1 << (bits - 1)) - 1;
    long long r = (long long)nearbyint(smp * (double)obd * coeff);
    int16_t s = (int16_t)r;           /* SmallInt assignment, range checks off */
    if (neg) s = (int16_t)(-s);
    if (s < -obd + 1) s = (int16_t)(-obd + 1);
    if (s > obd - 1) s = (int16_t)(obd - 1);
    return s;
}

/* enc:1665-1680 makeFloatSample(5 args) */
double gsc_ref_dequant(int16_t q, int bits, int atten, int neg, double law)
{
    double coeff = atten_coeff(atten, law);
    double obd = (double)((1 << (bits - 1)) - 1);
    int16_t s = q;
    if (neg) s = (int16_t)(-s);
    double r = (double)s / (obd * coeff);
    if (r < -1.0) r = -1.0;
    if (r > 1.0) r = 1.0;
    return r;
}

/* enc:1682-1698 ComputeAttenuation */
int gsc_ref_attenuation(int cs, const double *x, double law)
{
    int hi = 0;
    for (int i = 0; i < cs; ++i) {
        int v = (int)ceil(fabs(x[i] * 32767.0));
        if (v > hi) hi = v;
    }
    int r = 0;
    double c = 1.0;
    do {
        ++r;
        c += (double)r * law;
    } while (!(((double)hi * c > 32767.0) || (r > GSC_MAX_ATTENUATION)));
    return r - 1;
}

/* ------------------------------------------------------------------ */
/* per chunk                                                          */
/* ------------------------------------------------------------------ */

/* enc:365-397 ComputeDstAttributes */
void gsc_ref_chunk_attrs(int cs, const double *x, double law,
                         int *atten, int *neg, int *rev)
{
    *atten = gsc_ref_attenuation(cs, x, law);
    double p1 = 0.0, p2 = 0.0;
    for (int i = 0; i < cs; ++i) if (x[i] < 0) p1 -= x[i];
    for (int i = 0; i < cs; ++i) if (x[i] > 0) p2 += x[i];
    *neg = p1 > p2;
    p1 = 0.0; p2 = 0.0;
    for (int i = 0; i < cs / 2; ++i) p1 += fabs(x[i]);
    for (int i = cs / 2; i < cs; ++i) p2 += fabs(x[i]);
    *rev = p1 > p2;
}

/* Trig tables: the same libm calls the reference's expressions make, hoisted
 * (cos/sin are pure, so hoisting does not change any value). */
typedef struct trig_tables {
    int cs;
    double *dct;   /* [k][n]  s_k folded later; cos(pi/cs*(n+0.5)*k)   enc:1712 */
    double *dc;    /* [k][i]  cos(-2*pi*k*i/N)                          enc:270 */
    double *ds;    /* [k][i]  sin(-2*pi*k*i/N)                          enc:271 */
    double *ic;    /* [k][i]  cos(2*pi*k*i/N)                           enc:292 */
    double *is;    /* [k][i]  sin(2*pi*k*i/N)                           enc:293 */
} trig_tables;

static void trig_init(trig_tables *t, int cs)
{
    t->cs = cs;
    t->dct = (double *)malloc(sizeof(double) * cs * cs * 5);
    t->dc = t->dct + cs * cs;
    t->ds = t->dc + cs * cs;
    t->ic = t->ds + cs * cs;
    t->is = t->ic + cs * cs;
    for (int k = 0; k < cs; ++k)
        for (int n = 0; n < cs; ++n) {
            t->dct[k * cs + n] = cos(GSC_PI / (double)cs * ((double)n + 0.5) * (double)k);
            t->dc[k * cs + n] = cos(-2.0 * GSC_PI * (double)k * (double)n / (double)cs);
            t->ds[k * cs + n] = sin(-2.0 * GSC_PI * (double)k * (double)n / (double)cs);
            t->ic[k * cs + n] = cos(2.0 * GSC_PI * (double)k * (double)n / (double)cs);
            t->is[k * cs + n] = sin(2.0 * GSC_PI * (double)k * (double)n / (double)cs);
        }
}
static void trig_free(trig_tables *t) { free(t->dct); }

/* enc:349-363 TChunk.ComputeDCT, enc:1700-1716, enc:258-322 */
static void chunk_features_t(const trig_tables *t, const double *x, int neg,
                             int rev, double *f)
{
    int cs = t->cs;
    double data[64], temp[64];
    for (int i = 0; i < cs; ++i)
        data[i] = x[rev ? cs - 1 - i : i] * (neg ? -1.0 : 1.0);   /* enc:356 */
    /* enc:1706-1715 orthonormal DCT-II */
    const double scale = sqrt(2.0 / (double)cs);
    for (int k = 0; k < cs; ++k) {
        double s = (k == 0) ? sqrt(0.5) : 1.0;
        double sum = 0;
        for (int n = 0; n < cs; ++n)
            sum += s * data[n] * t->dct[k * cs + n];
        f[k] = sum * scale;
    }
    /* enc:305-322 cepstrum: DFT power -> log10 -> |iDFT| */
    for (int k = 0; k < cs; ++k) {                                 /* enc:258-278 */
        double re = 0, im = 0;
        for (int i = 0; i < cs; ++i) {
            re += data[i] * t->dc[k * cs + i];
            im += data[i] * t->ds[k * cs + i];
        }
        temp[k] = re * re + im * im;
    }
    for (int i = 0; i < cs; ++i)                                   /* enc:316-318 */
        if (!(fabs(temp[i]) <= 1e-12))
            temp[i] = gsc_log_cr(temp[i]) * 0.43429448190325182765;
    for (int k = 0; k < cs; ++k) {                                 /* enc:280-302 */
        double re = 0, im = 0;
        for (int i = 0; i < cs; ++i) {
            re += temp[i] * t->ic[k * cs + i];
            im += temp[i] * t->is[k * cs + i];
        }
        re /= (double)cs;
        im /= (double)cs;
        data[k] = sqrt(re * re + im * im);
    }
    for (int i = 0; i < cs; ++i) f[cs + i] = data[i] * 0.00001;    /* enc:362 */
}

void gsc_ref_chunk_features(int cs, const double *x, int neg, int rev, double *f)
{
    trig_tables t;
    trig_init(&t, cs);
    chunk_features_t(&t, x, neg, rev, f);
    trig_free(&t);
}

/* ------------------------------------------------------------------ */
/* per frame: divider search, chunk construction                      */
/* ------------------------------------------------------------------ */

/* enc:566-605 FindAttenuationDivider */
int gsc_ref_find_attenuation_divider(const int16_t *pcm, int64_t stride, int C,
                                     int S, int cs, int bits, double *v_out)
{
    double tmp[64];
    int bestDiv = 1;
    double best = 3.40282346638528860e+38;           /* MaxSingle */
    for (int i = 1; i <= 64; ++i) {
        double law = 1.0 / (double)i;
        double v = 0;
        for (int j = 0; j < C; ++j)
            for (int k = 0; k < S / cs; ++k) {
                int pos = k * cs;
                for (int l = 0; l < cs; ++l)
                    tmp[l] = gsc_ref_float_sample(pcm[j * stride + pos + l]);
                int atten = gsc_ref_attenuation(cs, tmp, law);
                for (int l = 0; l < cs; ++l) {
                    int16_t os = gsc_ref_quant(tmp[l], bits, atten, 0, law);
                    double fs = gsc_ref_dequant(os, bits, atten, 0, law);
                    double d = tmp[l] - fs;
                    v += d * d;
                }
            }
        if (v_out) v_out[i - 1] = v;
        if (v < best) { best = v; bestDiv = i; }
    }
    return bestDiv;
}

/* enc:467-485 TBand.MakeChunks (+ enc:802-806 Single dataset) */
int gsc_ref_make_chunks(const int16_t *pcm, int64_t stride, int C, int S, int cs,
                        int bits, int divider, double *raw, uint8_t *attr,
                        uint8_t *atten, float *feat, int16_t *dst)
{
    double law = 1.0 / (double)divider;               /* enc:561-564 */
    int cc = (S - 1) / cs + 1;                        /* enc:455 */
    trig_tables t;
    trig_init(&t, cs);
    double x[64], f[128];
    for (int i = 0; i < cc; ++i)
        for (int ch = 0; ch < C; ++ch) {
            int n = i * C + ch;
            for (int l = 0; l < cs; ++l) {
                int p = i * cs + l;
                x[l] = (p < S) ? gsc_ref_float_sample(pcm[ch * stride + p]) : 0.0;
            }
            int a, ng, rv;
            gsc_ref_chunk_attrs(cs, x, law, &a, &ng, &rv);
            if (raw) memcpy(raw + (size_t)n * cs, x, sizeof(double) * cs);
            if (attr) attr[n] = (uint8_t)((ng << 1) | rv);
            if (atten) atten[n] = (uint8_t)a;
            if (dst)
                for (int l = 0; l < cs; ++l)
                    dst[(size_t)n * cs + l] = gsc_ref_quant(x[l], bits, a, ng, law);
            if (feat) {
                chunk_features_t(&t, x, ng, rv, f);
                for (int l = 0; l < 2 * cs; ++l)
                    feat[(size_t)n * 2 * cs + l] = (float)f[l];
            }
        }
    trig_free(&t);
    return cc * C;
}

/* ------------------------------------------------------------------ */
/* yakmo as called (enc:824-828); behaviour from yakmo_single.dll      */
/* ------------------------------------------------------------------ */

typedef struct xor128 { uint64_t x, y, z, w; } xor128;

/* init() RVA 0x18c4-0x18f3: Marsaglia xor128 on 64-bit lanes, then
 * u = (float)((double)w * 2^-64). */
static float xor128_gen(xor128 *g)
{
    uint64_t t = g->x ^ (g->x << 11);
    g->x = g->y; g->y = g->z; g->z = g->w;
    g->w = (g->w ^ (g->w >> 19)) ^ (t ^ (t >> 8));
    return (float)((double)g->w * 5.42101086242752217e-20 /* 2^-64 */);
}

/* yakmo point::calc_dist, Euclidean (init() RVA 0x1dca-0x1e1b):
 *   d = (c.norm + p.norm) + 0;  for k: d -= (p_k + p_k) * c_k   (all float) */
static inline float yakmo_dist(const float *p, float pnorm, const float *c,
                               float cnorm, int D)
{
    float d = cnorm + pnorm;
    d = d + 0.0f;
    for (int k = 0; k < D; ++k) {
        float t = p[k] + p[k];
        t = t * c[k];
        d = d - t;
    }
    return d;
}

void gsc_ref_yakmo(const float *X, int N, int D, int K, int init_type,
                   int max_iter, float *centroids, int32_t *labels,
                   int32_t *seeds_out)
{
    float *pnorm = (float *)malloc(sizeof(float) * N);
    float *up = (float *)malloc(sizeof(float) * N);
    float *lo = (float *)malloc(sizeof(float) * N);
    int32_t *id = (int32_t *)malloc(sizeof(int32_t) * N);
    float *r = (float *)calloc(N, sizeof(float));
    float *cen = (float *)malloc(sizeof(float) * (size_t)K * D);
    float *cnorm = (float *)malloc(sizeof(float) * K);
    float *sum = (float *)calloc((size_t)K * D, sizeof(float));
    int32_t *cnt = (int32_t *)calloc(K, sizeof(int32_t));
    uint8_t *chosen = (uint8_t *)calloc(N, 1);

    /* load (RVA 0x2b80 -> 0x1540): norm = sum v*v left to right in float */
    for (int j = 0; j < N; ++j) {
        float s = 0.0f;
        for (int k = 0; k < D; ++k) {
            float v = X[(size_t)j * D + k];
            float m = v * v;
            s = s + m;
        }
        pnorm[j] = s;
        up[j] = 0.0f; lo[j] = 0.0f; id[j] = 0;
    }

    xor128 g = { 123456789ull, 362436069ull, 521288629ull, 88675123ull };
    float obj = 0.0f;
    for (int i = 0; i < K; ++i) {
        uint32_t c;
        float u = xor128_gen(&g);
        if (init_type == 0 || i == 0) {
            /* RANDOM, or first k-means++ seed: floor(u * (float)N) */
            c = (uint32_t)(int64_t)floorf(u * (float)N);
        } else {
            /* std::lower_bound(r.begin(), r.end(), u * obj) */
            float target = u * obj;
            int64_t first = 0, count = N;
            while (count > 0) {
                int64_t half = count >> 1;
                if (target > r[first + half]) {
                    first = first + half + 1;
                    count = count - half - 1;
                } else
                    count = half;
            }
            c = (uint32_t)first;
        }
        /* linear probe past already chosen points (RVA 0x1b20-0x1bd8) */
        while (c < (uint32_t)N && chosen[c])
            c = (c >= (uint32_t)(N - 1)) ? 0u : c + 1u;
        if (c >= (uint32_t)N) c = (uint32_t)(N - 1);      /* RVA 0x1c50-0x1c5a */
        chosen[c] = 1;
        if (seeds_out) seeds_out[i] = (int32_t)c;
        memcpy(cen + (size_t)i * D, X + (size_t)c * D, sizeof(float) * D);
        cnorm[i] = pnorm[c];

        obj = 0.0f;
        for (int j = 0; j < N; ++j) {
            const float *p = X + (size_t)j * D;
            float d = yakmo_dist(p, pnorm[j], cen + (size_t)i * D, cnorm[i], D);
            if (i == 0 || up[j] > d) {
                lo[j] = up[j]; up[j] = d; id[j] = i;
            } else if (i == 1) {
                lo[j] = d;
            } else if (lo[j] > d) {
                lo[j] = d;
            }
            if (i < K - 1) {
                if (init_type == 1) { obj = obj + up[j]; r[j] = obj; }
            } else {
                /* last seed: add the point to its cell */
                float *s = sum + (size_t)id[j] * D;
                for (int k = 0; k < D; ++k) s[k] = p[k] + s[k];
                cnt[id[j]]++;
            }
        }
    }

    /* run() RVA 0x21d0: for (i = 0; i <= iter; ++i) { if moved: means;
     * if !moved break; reassign (sums updated incrementally) } */
    int64_t moved = N;
    for (int it = 0; it <= max_iter; ++it) {
        if (moved) {
            for (int c = 0; c < K; ++c) {
                float nrm = 0.0f;
                float fc = (float)cnt[c];
                for (int k = 0; k < D; ++k) {
                    float v = sum[(size_t)c * D + k] / fc;   /* 0/0 -> NaN */
                    float m = v * v;
                    nrm = m + nrm;
                    cen[(size_t)c * D + k] = v;
                }
                cnorm[c] = nrm;
            }
        }
        if (!moved) break;
        moved = 0;
        for (int j = 0; j < N; ++j) {
            const float *p = X + (size_t)j * D;
            int best = id[j];
            float bd = INFINITY;
            for (int c = 0; c < K; ++c) {     /* strict <: earliest centroid wins ties */
                float d = yakmo_dist(p, pnorm[j], cen + (size_t)c * D, cnorm[c], D);
                if (d < bd) { bd = d; best = c; }
            }
            if (best != id[j]) {
                float *so = sum + (size_t)id[j] * D, *sn = sum + (size_t)best * D;
                for (int k = 0; k < D; ++k) { so[k] = so[k] - p[k]; sn[k] = sn[k] + p[k]; }
                cnt[id[j]]--; cnt[best]++;
                id[j] = best;
                ++moved;
            }
        }
    }
    memcpy(centroids, cen, sizeof(float) * (size_t)K * D);
    if (labels) for (int j = 0; j < N; ++j) labels[j] = id[j];

    free(pnorm); free(up); free(lo); free(id); free(r); free(cen); free(cnorm);
    free(sum); free(cnt); free(chosen);
}

/* ------------------------------------------------------------------ */
/* exact nearest neighbour (ANN annkSearch, eps = 0)                   */
/* ------------------------------------------------------------------ */

/* ANN distance: d = 0; for k: t = q[k]-p[k]; d = d + t*t  (float, no FMA).
 * Ct is the codebook transposed [D][Kp] so the k loop vectorises; the
 * per-centroid operation order is unchanged. */
static void dist_all(const float *q, const float *Ct, int Kp, int K, int D,
                     float *acc)
{
    for (int k = 0; k < K; ++k) acc[k] = 0.0f;
    for (int d = 0; d < D; ++d) {
        const float *row = Ct + (size_t)d * Kp;
        float qd = q[d];
        for (int k = 0; k < K; ++k) {
            float t = qd - row[k];
            float m = t * t;
            acc[k] = acc[k] + m;
        }
    }
}

/* strict <: lowest index on ties, NaN distances never win; every distance NaN (an all-NaN codebook) -> centroid 0
 * at d = +inf, what the kernels report */
static inline int argmin_first(const float *acc, int K, float *bd)
{
    int best = 0;
    float b = INFINITY;
    for (int k = 0; k < K; ++k)
        if (acc[k] < b) { b = acc[k]; best = k; }
    *bd = b;
    return best;
}

static float *transpose_codebook(const float *C, int K, int D)
{
    float *Ct = (float *)malloc(sizeof(float) * (size_t)K * D);
    for (int k = 0; k < K; ++k)
        for (int d = 0; d < D; ++d) Ct[(size_t)d * K + k] = C[(size_t)k * D + d];
    return Ct;
}

void gsc_ref_assign(const float *X, int N, int D, const float *centroids, int K,
                    int32_t *labels, float *dist_out)
{
    float *Ct = transpose_codebook(centroids, K, D);
    float *acc = (float *)malloc(sizeof(float) * K);
    for (int j = 0; j < N; ++j) {
        float bd;
        dist_all(X + (size_t)j * D, Ct, K, K, D, acc);
        labels[j] = argmin_first(acc, K, &bd);
        if (dist_out) dist_out[j] = bd;
    }
    free(Ct); free(acc);
}

/* ------------------------------------------------------------------ */
/* enc:699-765 KNNScanReduce                                           */
/* ------------------------------------------------------------------ */

static int same_value_d(double a, double b, double eps)
{
    return (a > b) ? ((a - b) <= eps) : ((b - a) <= eps);
}

static double int_power10_neg(int prec)
{
    double p = 1.0, base = 10.0;
    for (int i = 0; i < prec; ++i) p *= base;
    return 1.0 / p;
}

int gsc_ref_knn_scan_reduce_batched(const float *X, int N, int D,
                                    float *centroids, int K, int precision,
                                    int max_passes, int batch, int32_t *labels,
                                    double *err_out)
{
    if (batch < 1) batch = 1;
    float *Ct = transpose_codebook(centroids, K, D);
    float *acc = (float *)malloc(sizeof(float) * K);
    int32_t *cnts[2];
    cnts[0] = (int32_t *)malloc(sizeof(int32_t) * K);
    cnts[1] = (int32_t *)malloc(sizeof(int32_t) * K);
    int32_t *bidx = (int32_t *)malloc(sizeof(int32_t) * batch);
    float *bdist = (float *)malloc(sizeof(float) * batch);
    for (int j = 0; j < K; ++j) { cnts[0][j] = 1; cnts[1][j] = 1; }   /* enc:717-721 */

    const double tol = int_power10_neg(precision);
    int iter = 0;
    double err = 3.40282346638528860e+38, prevErr;                     /* enc:724 */
    do {
        prevErr = err;
        err = 0;
        const int odd = iter & 1;
        for (int i0 = 0; i0 < N; i0 += batch) {
            int nb = (N - i0 < batch) ? (N - i0) : batch;
            for (int b = 0; b < nb; ++b) {                             /* enc:733 */
                dist_all(X + (size_t)(i0 + b) * D, Ct, K, K, D, acc);
                bidx[b] = argmin_first(acc, K, &bdist[b]);
            }
            for (int b = 0; b < nb; ++b) {
                int i = i0 + b, bi = bidx[b];
                /* enc:735 rate := 1 / sqrt(cnts[not Odd(iter), bestIdx]) */
                float rate = (float)(1.0 / sqrt((double)cnts[!odd][bi]));
                for (int k = 0; k < D; ++k) {                          /* enc:736-740 */
                    float c = Ct[(size_t)k * K + bi];
                    float v = X[(size_t)i * D + k] - c;
                    float m = v * rate;
                    Ct[(size_t)k * K + bi] = c + m;
                }
                labels[i] = bi;                                        /* enc:742 */
                err += (double)sqrtf(bdist[b] / (float)D);             /* enc:743 */
                cnts[odd][bi] += 1;                                    /* enc:744 */
            }
        }
        for (int j = 0; j < K; ++j) cnts[!odd][j] = 1;                /* enc:754-755 */
        ++iter;
    } while (!(same_value_d(err, prevErr, tol) || iter >= max_passes)); /* enc:761 */

    for (int k = 0; k < K; ++k)
        for (int d = 0; d < D; ++d) centroids[(size_t)k * D + d] = Ct[(size_t)d * K + k];
    if (err_out) *err_out = err;
    free(Ct); free(acc); free(cnts[0]); free(cnts[1]); free(bidx); free(bdist);
    return iter;
}

int gsc_ref_knn_scan_reduce(const float *X, int N, int D, float *centroids,
                            int K, int precision, int max_passes,
                            int32_t *labels, double *err_out)
{
    return gsc_ref_knn_scan_reduce_batched(X, N, D, centroids, K, precision,
                                           max_passes, 1, labels, err_out);
}

/* ------------------------------------------------------------------ */
/* ANN 1.1.2 kd-tree (D. Mount, S. Arya), restated from its published   */
/* source (kd_tree.cpp, kd_split.cpp, kd_util.cpp, kd_search.cpp): the  */
/* structure KNNScanReduce really searches.  enc:729 builds it over the */
/* centroid rows (bucket size 1, ANN_KD_STD) at the start of every pass */
/* and enc:733 asks for the nearest point (annkSearch, k = 1, eps = 0). */
/* ANN keeps the caller's row pointers (no copy, SURVEY.md 3.2): leaf   */
/* distances read the LIVE rows, which enc:736-740 moves between        */
/* queries, while splitting planes and bounding boxes date from the     */
/* start of the pass.  ANNcoord = ANNdist = float in the shipped DLL.   */
/* Ties keep the first point VISITED (ANNmin_k::insert), not the lowest */
/* index.  ANN.dll's source is not in the reference tree: third-party,  */
/* version string "ANN Version 1.1.2".                                  */
/* ------------------------------------------------------------------ */
static float knnfit_epsilon(int bits, double law);
static inline int same_value_f(float a, float b, float eps);
typedef struct ann_node { int cd; float cv, lo_b, hi_b; int lo, hi; int pt; } ann_node;   /* pt >= 0: leaf; -2: trivial */
typedef struct ann_tree {
    const float *pts; int dim, n;
    ann_node *nodes; int n_nodes, root;
    float *bb_lo, *bb_hi;
    int32_t *pidx;
} ann_tree;

#define ANN_PA(t, i, d) ((t)->pts[(size_t)(t)->pidx[(i)] * (t)->dim + (d)])

static int ann_max_spread(const ann_tree *t, int off, int n)        /* kd_util.cpp annMaxSpread / annSpread */
{
    int max_dim = 0;
    float max_spr = 0;
    if (n == 0) return max_dim;
    for (int d = 0; d < t->dim; ++d) {
        float mn = ANN_PA(t, off, d), mx = mn;
        for (int i = 1; i < n; ++i) {
            float c = ANN_PA(t, off + i, d);
            if (c < mn) mn = c; else if (c > mx) mx = c;
        }
        float spr = mx - mn;
        if (spr > max_spr) { max_spr = spr; max_dim = d; }
    }
    return max_dim;
}

static void ann_median_split(ann_tree *t, int off, int n, int d, float *cv, int n_lo)   /* kd_util.cpp annMedianSplit */
{
#define PAV(i) ANN_PA(t, off + (i), d)
#define PASWAP(a, b) do { int32_t tmp_ = t->pidx[off + (a)]; t->pidx[off + (a)] = t->pidx[off + (b)]; t->pidx[off + (b)] = tmp_; } while (0)
    int l = 0, r = n - 1;
    while (l < r) {
        int i = (r + l) / 2, k;
        if (PAV(i) > PAV(r)) PASWAP(i, r);
        PASWAP(l, i);
        float c = PAV(l);
        i = l; k = r;
        for (;;) {
            while (i < r && PAV(++i) < c) ;      /* (bounds added: NaN rows must not run off the array) */
            while (k > l && PAV(--k) > c) ;
            if (i < k) PASWAP(i, k); else break;
        }
        PASWAP(l, k);
        if (k > n_lo) r = k - 1;
        else if (k < n_lo) l = k + 1;
        else break;
    }
    if (n_lo > 0) {
        float c = PAV(0);
        int k = 0;
        for (int i = 1; i < n_lo; ++i) if (PAV(i) > c) { c = PAV(i); k = i; }
        PASWAP(n_lo - 1, k);
    }
    *cv = (float)(((double)PAV(n_lo - 1) + (double)PAV(n_lo)) / 2.0);
#undef PAV
#undef PASWAP
}

static int ann_build_rec(ann_tree *t, int off, int n)               /* kd_tree.cpp rkd_tree, bucket size 1 */
{
    int id = t->n_nodes++;
    ann_node *nd = &t->nodes[id];
    if (n <= 1) { nd->pt = (n == 0) ? -2 : t->pidx[off]; nd->lo = nd->hi = -1; return id; }
    int cd = ann_max_spread(t, off, n), n_lo = n / 2;                /* kd_split.cpp kd_split */
    float cv;
    ann_median_split(t, off, n, cd, &cv, n_lo);
    float lv = t->bb_lo[cd], hv = t->bb_hi[cd];
    t->bb_hi[cd] = cv;
    int lo = ann_build_rec(t, off, n_lo);
    t->bb_hi[cd] = hv;
    t->bb_lo[cd] = cv;
    int hi = ann_build_rec(t, off + n_lo, n - n_lo);
    t->bb_lo[cd] = lv;
    nd = &t->nodes[id];
    nd->pt = -1; nd->cd = cd; nd->cv = cv; nd->lo_b = lv; nd->hi_b = hv; nd->lo = lo; nd->hi = hi;
    return id;
}

static void ann_build(ann_tree *t, const float *pts, int n, int dim)
{
    t->pts = pts; t->n = n; t->dim = dim;
    t->nodes = (ann_node *)malloc(sizeof(ann_node) * (size_t)(2 * n + 2));
    t->n_nodes = 0;
    t->pidx = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    t->bb_lo = (float *)malloc(sizeof(float) * dim * 2);
    t->bb_hi = t->bb_lo + dim;
    for (int i = 0; i < n; ++i) t->pidx[i] = i;
    for (int d = 0; d < dim; ++d) {                                  /* annEnclRect */
        float lo = pts[d], hi = pts[d];
        for (int i = 0; i < n; ++i) {
            float c = pts[(size_t)i * dim + d];
            if (c < lo) lo = c; else if (c > hi) hi = c;
        }
        t->bb_lo[d] = lo; t->bb_hi[d] = hi;
    }
    t->root = ann_build_rec(t, 0, n);
}
static void ann_free(ann_tree *t) { free(t->nodes); free(t->pidx); free(t->bb_lo); }

typedef struct ann_query { const float *q; float best; int idx; long visited; } ann_query;

static void ann_search_rec(const ann_tree *t, int id, float box_dist, ann_query *s)   /* kd_search.cpp */
{
    const ann_node *nd = &t->nodes[id];
    if (nd->pt != -1) {                                              /* ANNkd_leaf::ann_search */
        if (nd->pt < 0) return;
        const float *pp = t->pts + (size_t)nd->pt * t->dim;
        float min_dist = s->best, dist = 0;
        int d;
        for (d = 0; d < t->dim; ++d) {
            float tt = s->q[d] - pp[d];
            float m = tt * tt;
            dist = dist + m;
            if (dist > min_dist) break;
        }
        if (d >= t->dim && s->idx < 0) { s->best = dist; s->idx = nd->pt; }             /* first point */
        else if (d >= t->dim && dist < s->best) { s->best = dist; s->idx = nd->pt; }    /* equal keys keep the first visited */
        s->visited++;
        return;
    }
    float cut_diff = s->q[nd->cd] - nd->cv;                          /* ANNkd_split::ann_search */
    if (cut_diff < 0) {
        ann_search_rec(t, nd->lo, box_dist, s);
        float box_diff = nd->lo_b - s->q[nd->cd];
        if (box_diff < 0) box_diff = 0;
        box_dist = box_dist + (cut_diff * cut_diff - box_diff * box_diff);
        if ((double)box_dist * 1.0 < (double)s->best) ann_search_rec(t, nd->hi, box_dist, s);
    } else {
        ann_search_rec(t, nd->hi, box_dist, s);
        float box_diff = s->q[nd->cd] - nd->hi_b;
        if (box_diff < 0) box_diff = 0;
        box_dist = box_dist + (cut_diff * cut_diff - box_diff * box_diff);
        if ((double)box_dist * 1.0 < (double)s->best) ann_search_rec(t, nd->lo, box_dist, s);
    }
}

static int ann_search1(const ann_tree *t, const float *q, float *dist_out, long *visited)
{
    float bd = 0;                                                    /* annBoxDistance */
    for (int d = 0; d < t->dim; ++d) {
        if (q[d] < t->bb_lo[d]) { float tt = t->bb_lo[d] - q[d]; bd = bd + tt * tt; }
        else if (q[d] > t->bb_hi[d]) { float tt = q[d] - t->bb_hi[d]; bd = bd + tt * tt; }
    }
    ann_query s = { q, 3.40282346638528860e+38f, -1, 0 };
    ann_search_rec(t, t->root, bd, &s);
    if (dist_out) *dist_out = s.best;
    if (visited) *visited += s.visited;
    return s.idx;
}

/* k nearest points, ascending by distance; equal keys keep the order they were visited in (ANNmin_k::insert).
 * enc:952 calls annkPriSearch, which visits the cells in another order than this (standard) search; for eps = 0
 * both return the same k distances, and the same rows wherever the k-th distance is not tied. */
typedef struct ann_kquery { const float *q; int k, n; float *key; int *idx; } ann_kquery;

static void ann_ksearch_rec(const ann_tree *t, int id, float box_dist, ann_kquery *s)
{
    const ann_node *nd = &t->nodes[id];
    if (nd->pt != -1) {
        if (nd->pt < 0) return;
        const float *pp = t->pts + (size_t)nd->pt * t->dim;
        float min_dist = (s->n == s->k) ? s->key[s->k - 1] : 3.40282346638528860e+38f, dist = 0;
        int d;
        for (d = 0; d < t->dim; ++d) {
            float tt = s->q[d] - pp[d];
            float m = tt * tt;
            dist = dist + m;
            if (dist > min_dist) break;
        }
        if (d >= t->dim) {                                       /* ANNmin_k::insert */
            int i;
            for (i = s->n; i > 0; --i) {
                if (s->key[i - 1] > dist) { if (i < s->k) { s->key[i] = s->key[i - 1]; s->idx[i] = s->idx[i - 1]; } }
                else break;
            }
            if (i < s->k) { s->key[i] = dist; s->idx[i] = nd->pt; }
            if (s->n < s->k) s->n++;
        }
        return;
    }
    float cut_diff = s->q[nd->cd] - nd->cv;
    int near_c = (cut_diff < 0) ? nd->lo : nd->hi, far_c = (cut_diff < 0) ? nd->hi : nd->lo;
    ann_ksearch_rec(t, near_c, box_dist, s);
    float box_diff = (cut_diff < 0) ? nd->lo_b - s->q[nd->cd] : s->q[nd->cd] - nd->hi_b;
    if (box_diff < 0) box_diff = 0;
    box_dist = box_dist + (cut_diff * cut_diff - box_diff * box_diff);
    float kth = (s->n == s->k) ? s->key[s->k - 1] : 3.40282346638528860e+38f;
    if ((double)box_dist * 1.0 < (double)kth) ann_ksearch_rec(t, far_c, box_dist, s);
}

/* enc:915-965 the way the binary runs it: ANN kd-tree over the 4R variant rows (enc:945), 64 nearest rows per
 * chunk (enc:952), lowest index within epsilon of the nearest (enc:954-958).  Same answers as gsc_ref_knnfit's
 * `best` wherever at most 64 rows lie inside the band. */
void gsc_ref_knnfit_kdtree(const int16_t *dict, const uint8_t *datten, int R, int cs, int bits, int divider,
                           const double *raw, int N, int32_t *best, int32_t *use)
{
    double law = 1.0 / (double)divider;
    int M = R * 4;
    float *V = (float *)malloc(sizeof(float) * (size_t)M * cs);
    gsc_ref_knnfit_variants(dict, datten, R, cs, bits, divider, V);
    ann_tree t;
    ann_build(&t, V, M, cs);
    float eps = knnfit_epsilon(bits, law);
    float key[GSC_BUCKET]; int idx[GSC_BUCKET]; float q[64];
    if (use) memset(use, 0, sizeof(int32_t) * R);
    int kk = M < GSC_BUCKET ? M : GSC_BUCKET;
    for (int i = 0; i < N; ++i) {
        for (int j = 0; j < cs; ++j) q[j] = (float)raw[(size_t)i * cs + j];
        float bd = 0;
        for (int d = 0; d < cs; ++d) {
            if (q[d] < t.bb_lo[d]) { float tt = t.bb_lo[d] - q[d]; bd = bd + tt * tt; }
            else if (q[d] > t.bb_hi[d]) { float tt = q[d] - t.bb_hi[d]; bd = bd + tt * tt; }
        }
        ann_kquery s = { q, kk, 0, key, idx };
        ann_ksearch_rec(&t, t.root, bd, &s);
        float a = sqrtf(key[0] / (float)cs);
        int b = idx[0];
        for (int j = 1; j < s.n; ++j)
            if (same_value_f(a, sqrtf(key[j] / (float)cs), eps) && idx[j] < b) b = idx[j];
        best[i] = b;
        if (use) use[b >> 2]++;
    }
    ann_free(&t);
    free(V);
}

/* enc:699-765 with the search the binary performs: an ANN kd-tree over the LIVE centroid rows, rebuilt at the
 * start of every pass (enc:729, 759).  mode 0: the tree as ANN uses it (planes and boxes go stale while the pass
 * moves the rows; ties to the first point visited) -- the closest this restatement gets to the shipped encoder.
 * stats (optional, 2 longs): points visited, queries whose answer differs from the exact nearest centroid. */
int gsc_ref_knn_scan_reduce_kdtree(const float *X, int N, int D, float *centroids, int K, int precision,
                                   int max_passes, int32_t *labels, double *err_out, long *stats)
{
    int32_t *cnts[2];
    cnts[0] = (int32_t *)malloc(sizeof(int32_t) * K);
    cnts[1] = (int32_t *)malloc(sizeof(int32_t) * K);
    for (int j = 0; j < K; ++j) { cnts[0][j] = 1; cnts[1][j] = 1; }
    const double tol = int_power10_neg(precision);
    int iter = 0;
    double err = 3.40282346638528860e+38, prevErr;
    long visited = 0, inexact = 0;
    float *acc = stats ? (float *)malloc(sizeof(float) * K) : NULL;
    do {
        prevErr = err;
        err = 0;
        const int odd = iter & 1;
        ann_tree t;
        ann_build(&t, centroids, K, D);                                /* enc:729 */
        for (int i = 0; i < N; ++i) {
            const float *x = X + (size_t)i * D;
            float best;
            int bi = ann_search1(&t, x, &best, &visited);              /* enc:733 */
            if (bi < 0) { bi = 0; best = 0; }
            if (stats) {            /* how often do the stale planes / the tie order change the answer? */
                float bd = INFINITY; int be = 0;
                for (int c = 0; c < K; ++c) {
                    float d = 0;
                    for (int k = 0; k < D; ++k) { float tt = x[k] - centroids[(size_t)c * D + k]; d = d + tt * tt; }
                    if (d < bd) { bd = d; be = c; }
                }
                inexact += (be != bi);
            }
            float rate = (float)(1.0 / sqrt((double)cnts[!odd][bi]));  /* enc:735 */
            float *c = centroids + (size_t)bi * D;
            for (int k = 0; k < D; ++k) { float v = x[k] - c[k]; float m = v * rate; c[k] = c[k] + m; }   /* enc:736-740 */
            labels[i] = bi;
            err += (double)sqrtf(best / (float)D);                     /* enc:743 */
            cnts[odd][bi] += 1;
        }
        for (int j = 0; j < K; ++j) cnts[!odd][j] = 1;
        ann_free(&t);                                                  /* enc:759 */
        ++iter;
    } while (!(same_value_d(err, prevErr, tol) || iter >= max_passes));
    if (err_out) *err_out = err;
    if (stats) { stats[0] = visited; stats[1] = inexact; }
    free(cnts[0]); free(cnts[1]); free(acc);
    return iter;
}

/* Plain batch Lloyd (the 1e-4 centroid contract of BASELINE.json).  There is no
 * Lloyd in the reference to follow (enc:824 calls yakmo with maxIter = 0), so the
 * arithmetic is ours: member rows are accumulated in Double and the mean is
 * rounded to Single once, which makes the result independent of the summation
 * order (up to a ~1e-9 chance per coordinate) -- the property the multi-GPU
 * split of one frame needs. */
void gsc_ref_lloyd(const float *X, int N, int D, float *centroids, int K,
                   int iters, int32_t *labels)
{
    double *sum = (double *)malloc(sizeof(double) * (size_t)K * D);
    int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * K);
    for (int it = 0; it < iters; ++it) {
        gsc_ref_assign(X, N, D, centroids, K, labels, NULL);
        memset(sum, 0, sizeof(double) * (size_t)K * D);
        memset(cnt, 0, sizeof(int32_t) * K);
        for (int j = 0; j < N; ++j) {
            double *s = sum + (size_t)labels[j] * D;
            for (int k = 0; k < D; ++k) s[k] = s[k] + (double)X[(size_t)j * D + k];
            cnt[labels[j]]++;
        }
        for (int c = 0; c < K; ++c)
            if (cnt[c] > 0)
                for (int k = 0; k < D; ++k)
                    centroids[(size_t)c * D + k] = (float)(sum[(size_t)c * D + k] / (double)cnt[c]);
    }
    gsc_ref_assign(X, N, D, centroids, K, labels, NULL);
    free(sum); free(cnt);
}

/* ------------------------------------------------------------------ */
/* FPC fgl TFPSList.QuickSort (rtl/objpas/fgl.pp), descending by key   */
/* ------------------------------------------------------------------ */

/* Compare(Item1, Item2) = CompareValue(Item2.key, Item1.key)  enc:775-783 */
static inline int cmp_inv(const int32_t *keys, int32_t a, int32_t b)
{
    int32_t ka = keys[a], kb = keys[b];
    return (kb < ka) ? -1 : (kb > ka) ? 1 : 0;
}

static void fpc_quicksort(const int32_t *keys, int32_t *items, int L, int R)
{
    int I, J, P;
    do {
        I = L; J = R;
        P = (int)(((uint32_t)L + (uint32_t)R) / 2u);
        do {
            int32_t pivot = items[P];
            while (cmp_inv(keys, pivot, items[I]) > 0) ++I;
            while (cmp_inv(keys, pivot, items[J]) < 0) --J;
            if (I <= J) {
                int32_t t = items[I]; items[I] = items[J]; items[J] = t;
                if (P == I) P = J; else if (P == J) P = I;
                ++I; --J;
            }
        } while (!(I > J));
        if (L < J) fpc_quicksort(keys, items, L, J);
        L = I;
    } while (!(I >= R));
}

void gsc_ref_fpc_sort_desc(const int32_t *keys, int32_t *perm, int n)
{
    if (n < 2) return;                 /* TFPSList.Sort: if FCount < 2 then exit */
    fpc_quicksort(keys, perm, 0, n - 1);
}

/* ------------------------------------------------------------------ */
/* enc:843-889 class means, population sort, dictionary quantisation   */
/* ------------------------------------------------------------------ */

static void quantise_entry(const float *mean, int cs, int bits, double law,
                           int16_t *dict, uint8_t *datten, uint8_t *dattr)
{
    double x[64];
    for (int k = 0; k < cs; ++k) {
        double v = (double)mean[k];
        x[k] = (v != v) ? 0.0 : v;                      /* nan0, enc:876 */
    }
    int a, ng, rv;
    gsc_ref_chunk_attrs(cs, x, law, &a, &ng, &rv);      /* enc:880 */
    for (int k = 0; k < cs; ++k)
        dict[k] = gsc_ref_quant(x[k], bits, a, ng, law); /* enc:881 */
    *datten = (uint8_t)a;
    *dattr = (uint8_t)((ng << 1) | rv);
}

void gsc_ref_build_dictionary(const int32_t *labels, const double *raw,
                              const uint8_t *attr, int N, int cs, int K,
                              int bits, int divider, float *means,
                              int32_t *order, int32_t *counts, int16_t *dict,
                              uint8_t *datten, uint8_t *dattr, int32_t *entry)
{
    double law = 1.0 / (double)divider;
    double *acc = (double *)calloc((size_t)K * cs, sizeof(double));
    int32_t *cnt = (int32_t *)calloc(K, sizeof(int32_t));
    float *m0 = (float *)malloc(sizeof(float) * (size_t)K * cs);
    /* enc:853-860: ascending j per cluster == one pass in j order */
    for (int j = 0; j < N; ++j) {
        int c = labels[j];
        int rv = attr[j] & 1, ng = (attr[j] >> 1) & 1;
        for (int k = 0; k < cs; ++k)
            acc[(size_t)c * cs + k] += raw[(size_t)j * cs + (rv ? cs - 1 - k : k)] * (ng ? -1.0 : 1.0);
        cnt[c]++;
    }
    for (int c = 0; c < K; ++c)
        for (int k = 0; k < cs; ++k) {
            double y = (double)cnt[c];
            double v = (fabs(y) <= 1e-12) ? 0.0 : acc[(size_t)c * cs + k] / y;  /* div0 */
            m0[(size_t)c * cs + k] = (float)v;                                   /* enc:863 */
        }
    for (int c = 0; c < K; ++c) order[c] = c;
    gsc_ref_fpc_sort_desc(cnt, order, K);                                        /* enc:865 */
    int32_t *inv = (int32_t *)malloc(sizeof(int32_t) * K);
    for (int i = 0; i < K; ++i) {
        int c = order[i];
        inv[c] = i;                                                              /* enc:878 */
        counts[i] = cnt[c];
        memcpy(means + (size_t)i * cs, m0 + (size_t)c * cs, sizeof(float) * cs);
        quantise_entry(means + (size_t)i * cs, cs, bits, law, dict + (size_t)i * cs,
                       datten + i, dattr + i);
    }
    if (entry) for (int j = 0; j < N; ++j) entry[j] = inv[labels[j]];           /* enc:884-885 */
    free(acc); free(cnt); free(m0); free(inv);
}

/* enc:891-912 */
void gsc_ref_passthrough_dictionary(const double *raw, int N, int cs, int bits,
                                    int divider, int16_t *dict, uint8_t *datten,
                                    uint8_t *dattr)
{
    double law = 1.0 / (double)divider;
    for (int i = 0; i < N; ++i) {
        int a, ng, rv;
        gsc_ref_chunk_attrs(cs, raw + (size_t)i * cs, law, &a, &ng, &rv);
        for (int k = 0; k < cs; ++k)
            dict[(size_t)i * cs + k] = gsc_ref_quant(raw[(size_t)i * cs + k], bits, a, ng, law);
        datten[i] = (uint8_t)a;
        dattr[i] = (uint8_t)((ng << 1) | rv);
    }
}

/* ------------------------------------------------------------------ */
/* enc:915-978 KNNFit                                                  */
/* ------------------------------------------------------------------ */

void gsc_ref_knnfit_variants(const int16_t *dict, const uint8_t *datten, int R,
                             int cs, int bits, int divider, float *V)
{
    double law = 1.0 / (double)divider;
    for (int i = 0; i < R * 2; ++i)                    /* enc:930-938 */
        for (int j = 0; j < cs; ++j) {
            int e = i >> 1, ng = i & 1;
            V[((size_t)i * 2 + 0) * cs + j] =
                (float)gsc_ref_dequant(dict[(size_t)e * cs + j], bits, datten[e], ng, law);
            V[((size_t)i * 2 + 1) * cs + j] =
                (float)gsc_ref_dequant(dict[(size_t)e * cs + cs - 1 - j], bits, datten[e], ng, law);
        }
}

static float knnfit_epsilon(int bits, double law)
{
    float maxLaw = 1.0f;                               /* enc:940-942 */
    for (int j = 0; j <= GSC_MAX_ATTENUATION; ++j)
        maxLaw = (float)((double)maxLaw + (double)j * law);
    float a = 1.0f / ((float)(1 << bits) * maxLaw);    /* enc:943 */
    double b = 1.0 / 32767.0;
    double m = ((double)a > b) ? (double)a : b;
    return (float)m;
}

static inline int same_value_f(float a, float b, float eps)
{
    return (a > b) ? ((a - b) <= eps) : ((b - a) <= eps);
}

typedef struct cand { float d; int32_t idx; } cand;
static int cand_cmp(const void *a, const void *b)
{
    const cand *x = (const cand *)a, *y = (const cand *)b;
    if (x->d < y->d) return -1;
    if (x->d > y->d) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);
}

float gsc_ref_knnfit(const int16_t *dict, const uint8_t *datten, int R, int cs,
                     int bits, int divider, const double *raw, int N,
                     int32_t *best, int32_t *use, int32_t *band,
                     int32_t *best_all, int32_t *dbl_diff)
{
    double law = 1.0 / (double)divider;
    int M = R * 4;
    float *V = (float *)malloc(sizeof(float) * (size_t)M * cs);
    gsc_ref_knnfit_variants(dict, datten, R, cs, bits, divider, V);
    float *Vt = transpose_codebook(V, M, cs);
    float *acc = (float *)malloc(sizeof(float) * M);
    cand *cl = (cand *)malloc(sizeof(cand) * M);
    float eps = knnfit_epsilon(bits, law);
    float q[64];
    if (use) memset(use, 0, sizeof(int32_t) * R);

    for (int i = 0; i < N; ++i) {
        for (int j = 0; j < cs; ++j) q[j] = (float)raw[(size_t)i * cs + j];      /* enc:949-950 */
        dist_all(q, Vt, M, M, cs, acc);
        float d0;
        (void)argmin_first(acc, M, &d0);
        /* enc:954-958: band test in Single:  |sqrt(e0/cs) - sqrt(ej/cs)| <= eps */
        float a = sqrtf(d0 / (float)cs);
        int nb = 0, ball = -1, bdbl = -1;
        double ad = sqrt((double)d0 / (double)cs);
        for (int v = 0; v < M; ++v) {
            float b = sqrtf(acc[v] / (float)cs);
            if (same_value_f(a, b, eps)) {
                if (ball < 0) ball = v;
                cl[nb].d = acc[v]; cl[nb].idx = v; ++nb;
            }
            if (bdbl < 0 && same_value_d(ad, sqrt((double)acc[v] / (double)cs), (double)eps))
                bdbl = v;
        }
        int b64 = ball;
        if (nb > GSC_BUCKET) {
            /* ANN returns only the 64 nearest rows (ascending d; equal d in
             * kd-tree visit order, which is not reproducible -> index order
             * here); the reference then takes the lowest index among them. */
            qsort(cl, nb, sizeof(cand), cand_cmp);
            b64 = cl[0].idx;
            for (int t = 1; t < GSC_BUCKET; ++t) if (cl[t].idx < b64) b64 = cl[t].idx;
        }
        best[i] = b64;
        if (use) use[b64 >> 2]++;                                               /* enc:962-964 */
        if (band) band[i] = nb;
        if (best_all) best_all[i] = ball;
        if (dbl_diff) dbl_diff[i] = (bdbl != ball);
    }
    free(V); free(Vt); free(acc); free(cl);
    return eps;
}

/* enc:970-977 */
int gsc_ref_finalize_dictionary(const int32_t *use, int R, int32_t *remap,
                                int32_t *new_order)
{
    int32_t *kept = (int32_t *)malloc(sizeof(int32_t) * (R > 0 ? R : 1));
    int n = 0;
    for (int i = 0; i < R; ++i) if (use[i] != 0) kept[n++] = i;  /* Delete keeps order */
    gsc_ref_fpc_sort_desc(use, kept, n);                         /* enc:974 */
    for (int i = 0; i < R; ++i) remap[i] = -1;
    for (int i = 0; i < n; ++i) { remap[kept[i]] = i; if (new_order) new_order[i] = kept[i]; }
    free(kept);
    return n;
}

/* ------------------------------------------------------------------ */
/* whole frame (enc:1433-1447 DoFrame)                                 */
/* ------------------------------------------------------------------ */

void gsc_ref_default_params(gsc_ref_params *p)
{
    p->chunk_size = 4;
    p->chunk_bit_depth = 8;
    p->chunks_per_frame = GSC_MAX_CHUNKS;
    p->precision = 3;
    p->max_passes = 100;
    p->kmeans_mode = 0;
    p->lloyd_iters = 30;
    p->batch = 512;
    p->frame_length_ms = 4000.0;
    p->vfr = 1.0;
    p->band_all = 0;
    p->reserved = 0;
}

int gsc_ref_encode_frame(const int16_t *pcm, int64_t stride, int C, int S,
                         const gsc_ref_params *p, gsc_ref_frame_out *out)
{
    const int cs = p->chunk_size, bits = p->chunk_bit_depth, K = p->chunks_per_frame;
    memset(out, 0, sizeof(*out));
    int divider = gsc_ref_find_attenuation_divider(pcm, stride, C, S, cs, bits, NULL);
    int cc = (S - 1) / cs + 1;
    int N = cc * C;
    double *raw = (double *)malloc(sizeof(double) * (size_t)N * cs);
    uint8_t *attr = (uint8_t *)malloc(N);
    uint8_t *atten = (uint8_t *)malloc(N);
    float *feat = (float *)malloc(sizeof(float) * (size_t)N * 2 * cs);
    gsc_ref_make_chunks(pcm, stride, C, S, cs, bits, divider, raw, attr, atten, feat, NULL);

    int R;
    int16_t *dict; uint8_t *datten, *dattr;
    out->passes = 0; out->err = 0;
    if (p->precision > 0 && N > K) {                       /* enc:808 */
        const int D = 2 * cs;
        float *cen = (float *)calloc((size_t)K * D, sizeof(float));
        int32_t *labels = (int32_t *)malloc(sizeof(int32_t) * N);
        gsc_ref_yakmo(feat, N, D, K, 1, 0, cen, labels, NULL);     /* enc:824-828 */
        if (p->kmeans_mode == 1) {
            gsc_ref_lloyd(feat, N, D, cen, K, p->lloyd_iters, labels);
            out->passes = p->lloyd_iters;
        } else {
            int batch = (p->kmeans_mode == 2) ? p->batch : 1;
            if (p->kmeans_mode == 3)
                out->passes = gsc_ref_knn_scan_reduce_kdtree(feat, N, D, cen, K, p->precision,
                                                             p->max_passes, labels, &out->err, NULL);
            else
                out->passes = gsc_ref_knn_scan_reduce_batched(feat, N, D, cen, K, p->precision,
                                                              p->max_passes, batch, labels, &out->err);
        }
        R = K;
        dict = (int16_t *)malloc(sizeof(int16_t) * (size_t)R * cs);
        datten = (uint8_t *)malloc(R); dattr = (uint8_t *)malloc(R);
        float *means = (float *)malloc(sizeof(float) * (size_t)K * cs);
        int32_t *order = (int32_t *)malloc(sizeof(int32_t) * K);
        int32_t *counts = (int32_t *)malloc(sizeof(int32_t) * K);
        gsc_ref_build_dictionary(labels, raw, attr, N, cs, K, bits, divider, means, order,
                                 counts, dict, datten, dattr, NULL);
        free(means); free(order); free(counts); free(cen); free(labels);
    } else {
        R = N;
        dict = (int16_t *)malloc(sizeof(int16_t) * (size_t)R * cs);
        datten = (uint8_t *)malloc(R); dattr = (uint8_t *)malloc(R);
        gsc_ref_passthrough_dictionary(raw, N, cs, bits, divider, dict, datten, dattr);
    }

    int32_t *best = (int32_t *)malloc(sizeof(int32_t) * N);
    int32_t *use = (int32_t *)malloc(sizeof(int32_t) * R);
    int32_t *band = (int32_t *)malloc(sizeof(int32_t) * N);
    if (p->kmeans_mode == 3 && !p->band_all) {
        gsc_ref_knnfit_kdtree(dict, datten, R, cs, bits, divider, raw, N, best, use);
        for (int j = 0; j < N; ++j) band[j] = 0;       /* (band populations are not computed in this mode) */
    } else if (p->band_all) {
        int32_t *b64 = (int32_t *)malloc(sizeof(int32_t) * N);
        gsc_ref_knnfit(dict, datten, R, cs, bits, divider, raw, N, b64, NULL, band, best, NULL);
        memset(use, 0, sizeof(int32_t) * R);
        for (int j = 0; j < N; ++j) use[best[j] >> 2]++;
        free(b64);
    } else
        gsc_ref_knnfit(dict, datten, R, cs, bits, divider, raw, N, best, use, band, NULL, NULL);
    int32_t *remap = (int32_t *)malloc(sizeof(int32_t) * R);
    int32_t *norder = (int32_t *)malloc(sizeof(int32_t) * R);
    int R2 = gsc_ref_finalize_dictionary(use, R, remap, norder);

    out->N = N; out->R = R2; out->divider = divider;
    out->dict = (int16_t *)malloc(sizeof(int16_t) * (size_t)(R2 > 0 ? R2 : 1) * cs);
    out->datten = (uint8_t *)malloc(R2 > 0 ? R2 : 1);
    for (int i = 0; i < R2; ++i) {
        memcpy(out->dict + (size_t)i * cs, dict + (size_t)norder[i] * cs, sizeof(int16_t) * cs);
        out->datten[i] = datten[norder[i]];
    }
    out->index = (int32_t *)malloc(sizeof(int32_t) * N);
    out->attr = (uint8_t *)malloc(N);
    out->overfull = 0;
    for (int j = 0; j < N; ++j) {
        out->index[j] = remap[best[j] >> 2];
        out->attr[j] = (uint8_t)(best[j] & 3);
        if (band[j] > GSC_BUCKET) out->overfull++;
    }
    free(raw); free(attr); free(atten); free(feat); free(dict); free(datten); free(dattr);
    free(best); free(use); free(band); free(remap); free(norder);
    return 0;
}

void gsc_ref_free_frame(gsc_ref_frame_out *out)
{
    free(out->dict); free(out->datten); free(out->index); free(out->attr);
    memset(out, 0, sizeof(*out));
}

/* ------------------------------------------------------------------ */
/* enc:1374-1425 frame cut                                             */
/* ------------------------------------------------------------------ */

int gsc_ref_plan_frames(const int16_t *pcm, int64_t stride, int C, int64_t S,
                        int sample_rate, const gsc_ref_params *p,
                        int64_t *starts, int max_frames)
{
    const int block = p->chunk_size;                   /* enc:1312-1315, underSample 1, blend 0 */
    int frameCount = (int)ceil((double)S / ((double)sample_rate * (p->frame_length_ms / 1000.0)));
    double avg = 0.0;
    for (int j = 0; j < C; ++j)
        for (int64_t i = 0; i < S; ++i) {
            double x = gsc_ref_float_sample(pcm[j * stride + i]);
            avg += x * x;
        }
    avg = sqrt(avg / ((double)S * (double)C));
    double total = 0.0;
    for (int64_t i = 0; i < S; ++i) {
        double smp = 0.0;
        for (int j = 0; j < C; ++j) {
            double x = gsc_ref_float_sample(pcm[j * stride + i]);
            smp += x * x;
        }
        smp = sqrt(smp / (double)C);
        total += 1.0 - (avg + (smp - avg) * p->vfr);   /* lerp enc:229-232 */
    }
    double per = total / (double)frameCount;
    int k = 0;
    int64_t nextStart = 0;
    double cur = 0.0;
    for (int64_t i = 0; i < S; ++i) {
        double smp = 0.0;
        for (int j = 0; j < C; ++j) {
            double x = gsc_ref_float_sample(pcm[j * stride + i]);
            smp += x * x;
        }
        smp = sqrt(smp / (double)C);
        cur += 1.0 - (avg + (smp - avg) * p->vfr);
        if ((i % block == 0) && (cur >= per)) {        /* enc:1411 */
            if (k < max_frames) starts[k] = nextStart;
            cur = 0.0; nextStart = i; ++k;
        }
    }
    if (k < max_frames) starts[k] = nextStart;
    ++k;
    return k;
}

/* ------------------------------------------------------------------ */
/* enc:980-1107 SaveStream                                             */
/* ------------------------------------------------------------------ */

typedef struct wr { uint8_t *buf; int64_t cap, pos; } wr;
static void w8(wr *w, unsigned v) { if (w->buf && w->pos < w->cap) w->buf[w->pos] = (uint8_t)v; w->pos++; }
static void w16(wr *w, unsigned v) { w8(w, v & 0xff); w8(w, (v >> 8) & 0xff); }
static void w32(wr *w, uint32_t v) { w16(w, v & 0xffff); w16(w, v >> 16); }

static int bsr_word(unsigned v) { int r = 0; while (v >>= 1) ++r; return r; }
static int vcbs(int index) { return index == 0 ? 0 : bsr_word((unsigned)index) / 3; }

int64_t gsc_ref_write_frame(const gsc_ref_frame_out *f, int C, int cs, int bits,
                            int sample_rate, uint8_t *buf, int64_t cap)
{
    wr w = { buf, cap, 0 };
    w16(&w, ((unsigned)C << 8) | 1u);                    /* enc:988-989 CStreamVersion = 1 */
    w16(&w, (unsigned)f->R);                             /* enc:990-991 CBandCount-1 = 0 */
    w16(&w, ((unsigned)cs << 8) | (unsigned)bits);       /* enc:992-993 */
    w32(&w, (uint32_t)sample_rate);                      /* enc:994-995 ChunkBlend 0 */
    w16(&w, (unsigned)f->divider);                       /* enc:996-997 */
    for (int j = 0; j < f->R / 2; ++j)                   /* enc:1003-1008 */
        w8(&w, ((unsigned)f->datten[j * 2] << 4) | f->datten[j * 2 + 1]);
    if (f->R & 1) w8(&w, (unsigned)f->datten[f->R - 1] << 4);
    if (bits == 8) {                                     /* enc:1015-1018 */
        for (int j = 0; j < f->R; ++j)
            for (int k = 0; k < cs; ++k)
                w8(&w, (unsigned)(f->dict[(size_t)j * cs + k] + 128) & 0xff);
    } else {                                             /* enc:1019-1039 */
        for (int j = 0; j < f->R; ++j) {
            for (int k = 0; k < cs / 2; ++k) {
                int s1 = f->dict[(size_t)j * cs + k * 2] + 2048;
                int s2 = f->dict[(size_t)j * cs + k * 2 + 1] + 2048;
                w8(&w, ((s1 >> 4) & 0xf0) | ((s2 >> 8) & 0x0f));
                w8(&w, s1 & 0xff);
                w8(&w, s2 & 0xff);
            }
            if (cs & 1) {
                int s1 = f->dict[(size_t)j * cs + cs - 1] + 2048;
                w8(&w, (s1 >> 4) & 0xf0);
                w8(&w, s1 & 0xff);
            }
        }
    }
    w32(&w, (uint32_t)(f->N / C));                       /* enc:1048 */
    int bitCnt = 0;
    uint32_t bitsacc = 0;
    for (int j = 0; j < f->N; ++j) {                     /* enc:1052-1098 */
        int idx = f->index[j];
        int vc = vcbs(idx);
        int pv = (j >= 1) ? vcbs(f->index[j - 1]) : -1;
        uint32_t code = 0; int sz = 0;
        code |= (uint32_t)((f->attr[j] >> 1) & 1) << sz; sz += 1;   /* Negative */
        code |= (uint32_t)(f->attr[j] & 1) << sz; sz += 1;          /* Reversed */
        if (vc == pv) { sz += 1; }
        else { code |= 1u << sz; sz += 1; code |= (uint32_t)vc << sz; sz += 2; }
        for (int k = vc; k >= 0; --k) {
            code |= (uint32_t)((idx >> (k * 3)) & 7) << sz; sz += 3;
        }
        bitsacc |= code << bitCnt;
        bitCnt += sz;
        if (bitCnt >= 16) { bitCnt -= 16; w16(&w, bitsacc & 0xffff); bitsacc >>= 16; }
    }
    if (bitCnt > 0) w16(&w, bitsacc & 0xffff);           /* enc:1100-1105 */
    return w.pos;
}

/* ------------------------------------------------------------------ */
/* dec:37-220 GSCUnpack                                                */
/* ------------------------------------------------------------------ */

int64_t gsc_ref_decode(const uint8_t *g, int64_t len, int16_t *out,
                       int64_t cap_samples, int *channels, int *sample_rate)
{
    const int32_t attrMul = (int32_t)nearbyint(32768.0 * (32767.0 / 2047.0));   /* dec:6 */
    int64_t pos = 0, written = 0;
    int C = 0;
    while (pos != len) {
        if (pos + 14 > len) return -1;
        /* dec:76-84 */
        pos += 1;                                   /* StreamVersion */
        int version = g[pos - 1];
        C = g[pos++];
        int R = (g[pos] | (g[pos + 1] << 8)) & 0x1fff; pos += 2;
        int bits = g[pos++];
        int cs = g[pos++];
        uint32_t sr = (uint32_t)g[pos] | ((uint32_t)g[pos + 1] << 8) | ((uint32_t)g[pos + 2] << 16) | ((uint32_t)g[pos + 3] << 24);
        pos += 4;
        int blend = (int)(sr >> 24); sr &= 0xffffff;
        int divider = g[pos] | (g[pos + 1] << 8); pos += 2;
        if (blend != 0 || cs <= 0 || cs > 64) return -1;
        if (channels) *channels = C;
        if (sample_rate) *sample_rate = (int)sr;
        int32_t lut[2][16];
        double law = 1.0 / (double)divider, lawAcc = 1.0;       /* dec:88-96 */
        for (int i = 0; i <= 15; ++i) {
            lawAcc += law * (double)i;
            lut[0][i] = (int32_t)nearbyint((double)attrMul / lawAcc);
            lut[1][i] = -lut[0][i];
        }
        uint8_t *att = (uint8_t *)malloc(R > 0 ? R : 1);
        int16_t *ch = (int16_t *)malloc(sizeof(int16_t) * (size_t)(R > 0 ? R : 1) * cs);
        for (int i = 0; i < R / 2; ++i) {                        /* dec:115-120 */
            int b = g[pos++];
            att[i * 2] = (uint8_t)((b & 0xf0) >> 4); att[i * 2 + 1] = (uint8_t)(b & 0x0f);
        }
        if (R & 1) { int b = g[pos++]; att[R - 1] = (uint8_t)((b & 0xf0) >> 4); }
        if (bits == 8) {                                         /* dec:131-137 */
            for (int i = 0; i < R; ++i)
                for (int j = 0; j < cs; ++j) {
                    int b = g[pos++];
                    ch[(size_t)i * cs + j] = (int16_t)(((b - 128) * 2047) / 127);
                }
        } else if (bits == 12) {                                 /* dec:138-158 */
            for (int i = 0; i < R; ++i) {
                for (int j = 0; j < cs / 2; ++j) {
                    int b = g[pos++];
                    int s1 = g[pos++] | ((b & 0xf0) << 4);
                    int s2 = g[pos++] | ((b & 0x0f) << 8);
                    ch[(size_t)i * cs + j * 2] = (int16_t)(s1 - 2048);
                    ch[(size_t)i * cs + j * 2 + 1] = (int16_t)(s2 - 2048);
                }
                if (cs & 1) {
                    int b = g[pos++];
                    int s1 = g[pos++] | ((b & 0xf0) << 4);
                    ch[(size_t)i * cs + cs - 1] = (int16_t)(s1 - 2048);
                }
            }
        } else { free(att); free(ch); return -1; }
        uint32_t flen = (uint32_t)g[pos] | ((uint32_t)g[pos + 1] << 8) | ((uint32_t)g[pos + 2] << 16) | ((uint32_t)g[pos + 3] << 24);
        pos += 4;                                                /* dec:164 */
        uint32_t bitsacc = 0; int bitCount = 0; int header = -1;
        int idx[16], ng[16], rv[16];
        for (uint32_t i = 0; i < flen; ++i) {
            for (int k = 0; k < C; ++k) {
#define FILLBITS() do { if (bitCount < 16 && pos < len) { uint32_t w = g[pos] | ((pos + 1 < len) ? ((uint32_t)g[pos + 1] << 8) : 0u); pos += 2; bitsacc |= w << bitCount; bitCount += 16; } } while (0)
#define GETBITS(n, dst) do { (dst) = (int)(bitsacc & ((1u << (n)) - 1)); bitsacc >>= (n); bitCount -= (n); } while (0)
                FILLBITS();
                GETBITS(1, ng[k]);
                rv[k] = 0;
                if (version > 0) GETBITS(1, rv[k]);
                int nh; GETBITS(1, nh);
                if (nh) GETBITS(2, header);
                FILLBITS();
                idx[k] = 0;
                for (int j = 0; j <= header; ++j) { int t; GETBITS(3, t); idx[k] = (idx[k] << 3) | t; }
            }
            for (int j = 0; j < cs; ++j)                          /* dec:195-202 */
                for (int k = 0; k < C; ++k) {
                    int32_t attr = lut[ng[k]][att[idx[k]]];
                    int32_t smp = ch[(size_t)idx[k] * cs + (rv[k] ? cs - 1 - j : j)];
                    uint32_t prod = (uint32_t)(attr * smp);
                    int16_t o = (int16_t)((prod >> 15) & 0xffff);
                    if (out && written < cap_samples * C) out[written] = o;
                    ++written;
                }
        }
        if (bitCount >= 16) { pos -= 2; bitCount -= 16; }         /* dec:205-209 */
        free(att); free(ch);
    }
    return C ? written / C : 0;
}

/* ------------------------------------------------------------------ */
/* enc:487-522 + 1518-1582 reconstruction; enc:1862-1880 PsyADelta     */
/* ------------------------------------------------------------------ */

void gsc_ref_reconstruct_frame(const gsc_ref_frame_out *f, int C, int S, int cs,
                               int bits, int16_t *out, int64_t stride)
{
    double law = 1.0 / (double)f->divider;
    int cc = f->N / C;
    for (int i = 0; i < cc; ++i)
        for (int chn = 0; chn < C; ++chn) {
            int n = i * C + chn;
            int e = f->index[n];
            int ng = (f->attr[n] >> 1) & 1, rv = f->attr[n] & 1;
            for (int j = 0; j < cs; ++j) {
                int p = i * cs + j;
                if (p >= S) continue;
                double smp = gsc_ref_dequant(f->dict[(size_t)e * cs + (rv ? cs - 1 - j : j)],
                                             bits, f->datten[e], ng, law);   /* enc:510 */
                out[chn * stride + p] = gsc_ref_make16(smp);                 /* enc:1580 */
            }
        }
}

double gsc_ref_psy_a_delta(const int16_t *a, const int16_t *b, int64_t n)
{
    double r = 0.0;                                   /* enc:1803-1814 on Double copies */
    for (int64_t i = 0; i < n; ++i) {
        double d = (double)a[i] - (double)b[i];
        r += d * d;
    }
    return sqrt(r / (double)n);
}

double gsc_ref_snr_db(const int16_t *ref, const int16_t *tst, int64_t n)
{
    double s = 0.0, e = 0.0;
    for (int64_t i = 0; i < n; ++i) {
        double x = (double)ref[i], d = x - (double)tst[i];
        s += x * x; e += d * d;
    }
    if (e == 0.0) return INFINITY;
    return 10.0 * log10(s / e);
}
