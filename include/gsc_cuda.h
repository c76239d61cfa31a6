/*
 * gsc_cuda.h -- C ABI of libgsc_cuda.so, the B200 (sm_100a) implementation of
 * the SoundChunks encoder hot path.
 *
 * The library drops in where encoder/extern.pas binds yakmo_single.dll and
 * ANN.dll today.  Citations: ext:L = /root/reference/encoder/extern.pas line L,
 * enc:L = /root/reference/encoder/encoder.lpr line L.
 *
 * Three groups of entry points:
 *   1. the legacy symbols, names/arity exactly as ext:112-123 (on x86-64 SysV
 *      `stdcall` and `cdecl` are the same convention);
 *   2. batched per-frame stages: one call replaces one loop of enc:566-978;
 *   3. gsc_encode_frames: whole DoFrame (enc:1433-1447) for a batch of
 *      independent frames on one GPU -- the unit that is sharded across GPUs.
 *
 * All pointers are HOST pointers unless the name ends in `_dev`.  There is no
 * CPU fallback: every call fails (non-zero / NULL / -1, gsc_last_error() set)
 * when no sm_100 device is usable.  Nothing throws or aborts across the ABI;
 * MXCSR is saved, masked and restored around every entry because the
 * FreePascal host runs with FP exceptions unmasked.
 *
 * Layouts:
 *   pcm       int16 planar [C][S]  (row stride in samples)
 *   chunk n   = i*C + ch, cs samples                      enc:475-484
 *   attr      bit0 Reversed | bit1 Negative               enc:960-961
 *   features  float [N][2*cs]                              enc:802-806
 *   variant   row = entry*4 + neg*2 + rev                  enc:928-938
 */
#ifndef GSC_CUDA_H
#define GSC_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSC_OK 0
#define GSC_ERR_CUDA 1
#define GSC_ERR_ARG 2
#define GSC_ERR_NODEVICE 3
#define GSC_ERR_UNSUPPORTED 4

/* ===================================================================== */
/* 1. Legacy ABI (ext:112-123)                                            */
/* ===================================================================== */

/* ext:112  yakmo_create(k, restartCount, maxIter, initType, initSeed,
 *          doNormalize, isVerbose).  initType 0 random / 1 k-means++;
 *          initSeed is a flag (0 = fixed xor128 seeds); doNormalize must be 0. */
void *yakmo_create(uint32_t k, uint32_t restartCount, int32_t maxIter,
                   int32_t initType, int32_t initSeed, int32_t doNormalize,
                   int32_t isVerbose);
/* ext:113 */
void yakmo_destroy(void *ay);
/* ext:114  dataset = rowCount row pointers of colCount floats (copied). */
void yakmo_load_train_data(void *ay, uint32_t rowCount, uint32_t colCount,
                           float **dataset);
/* ext:115  seeding + run(maxIter); writes one label per row. */
void yakmo_train_on_data(void *ay, int32_t *pointToCluster);
/* ext:116  writes k rows of colCount floats into caller-owned rows. */
void yakmo_get_centroids(void *ay, float **centroids);

/* ext:118  pa = n row pointers of dd floats.  Like ANN, the handle KEEPS the
 *          caller's row pointers (they must stay valid until destroy): before
 *          every query the rows are re-read and whatever changed is uploaded, so
 *          the enc:725-746 loop, which moves Centroids[bestIdx] between queries
 *          on one tree, sees its own updates.  bs and split are kd-tree hints
 *          and are ignored by the exact GPU search (no stale planes either). */
void *ann_kdtree_create(float **pa, int32_t n, int32_t dd, int32_t bs,
                        int32_t split);
/* ext:119  destroy(NULL) is a no-op. */
void ann_kdtree_destroy(void *akd);
/* ext:120  returns the index of the nearest point, *err = squared L2.
 *          eps must be 0 (exact search).  -1 on failure. */
int32_t ann_kdtree_search(void *akd, float *q, float eps, float *err);
/* ext:121 */
int32_t ann_kdtree_pri_search(void *akd, float *q, float eps, float *err);
/* ext:122  cnt nearest, ascending by (distance, index). */
void ann_kdtree_search_multi(void *akd, int32_t *idxs, float *errs, int32_t cnt,
                             float *q, float eps);
/* ext:123 */
void ann_kdtree_pri_search_multi(void *akd, int32_t *idxs, float *errs,
                                 int32_t cnt, float *q, float eps);

/* ===================================================================== */
/* Library / context                                                      */
/* ===================================================================== */

typedef struct gsc_ctx gsc_ctx;

/* Last error text of the calling thread ("" if none). */
const char *gsc_last_error(void);
/* Number of usable sm_100 devices (0 if none / no driver). */
int gsc_device_count(void);
/* One context = one device + one stream + scratch.  device < 0: round-robin
 * over the visible devices (this is how frames spread over GPUs when the
 * unmodified multi-threaded host drives the legacy ABI, mtprocs.pas:598). */
gsc_ctx *gsc_create(int device);
void gsc_destroy(gsc_ctx *ctx);
int gsc_ctx_device(const gsc_ctx *ctx);
/* cudaStream_t of the context, for callers that time with CUDA events. */
void *gsc_ctx_stream(const gsc_ctx *ctx);
int gsc_synchronize(gsc_ctx *ctx);

typedef struct gsc_stats {
    uint64_t kernel_launches;   /* kernels launched by this context */
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    double   last_stage_ms[8];  /* gsc_encode_frames: divider, chunks, seed,
                                   kmeans, dictionary, knnfit, finalize, total
                                   (CUDA events on the context stream) */
} gsc_stats;
int gsc_get_stats(gsc_ctx *ctx, gsc_stats *out);
/* Large batches run on two internal streams (even / odd frames); last_stage_ms adds both lanes up.
 * gsc_stage_busy_ms gives the wall-clock time during which stage `stage` (index into last_stage_ms, 0..6)
 * of the last batch ran on at least one of them (union of the two intervals; call after gsc_fetch_results). */
int gsc_stage_busy_ms(gsc_ctx *ctx, int stage, double *ms_out);
int gsc_reset_stats(gsc_ctx *ctx);

/* ===================================================================== */
/* 2. Batched per-frame stages (host buffers)                             */
/* ===================================================================== */

/* enc:566-605 FindAttenuationDivider.  v_out: optional double[64]. */
int gsc_find_attenuation_divider(gsc_ctx *ctx, const int16_t *pcm,
                                 int64_t stride, int C, int S, int cs, int bits,
                                 int *divider_out, double *v_out);

/* enc:467-485 MakeChunks (+ Single dataset enc:802-806).
 * Any output may be NULL.  atten/dst are the per-chunk attenuation and
 * quantised copy (enc:370, 432-439). */
int gsc_make_chunks(gsc_ctx *ctx, const int16_t *pcm, int64_t stride, int C,
                    int S, int cs, int bits, int divider, uint8_t *attr,
                    uint8_t *atten, float *feat, int16_t *dst);

/* yakmo as called at enc:824-828 on contiguous data: seeding + run(max_iter).
 * centroids float[K][D]; labels (optional) int32[N]; seeds (optional) int32[K]. */
int gsc_yakmo(gsc_ctx *ctx, const float *X, int N, int D, int K, int init_type,
              int max_iter, float *centroids, int32_t *labels, int32_t *seeds);

/* enc:699-765 KNNScanReduce: the reference's online rule, one point at a
 * time against the live centroids (exact NN, lowest index on ties).
 * centroids in/out; labels out; *passes, *err optional. */
int gsc_knn_scan_reduce(gsc_ctx *ctx, const float *X, int N, int D,
                        float *centroids, int K, int precision, int max_passes,
                        int32_t *labels, int *passes, double *err);

/* kmeans_mode 3: enc:699-765 with the search the reference binary performs -- an ANN 1.1.2 kd-tree over the
 * centroids, rebuilt at the start of every pass (planes and boxes from the pass start, leaves read the live rows,
 * ties to the first point visited).  Bit-identical to the oracle's kd-tree rule.  D in {4, 8},
 * 1 <= K <= 4096.  Same arguments as gsc_knn_scan_reduce. */
int gsc_knn_scan_reduce_kdtree(gsc_ctx *ctx, const float *X, int N, int D, float *centroids, int K, int precision,
                               int max_passes, int32_t *labels, int *passes, double *err);

/* Plain batch Lloyd (BASELINE.json's 1e-4 centroid contract): `iters` x
 * (exact assign, mean), then a final assign.  centroids in/out.  Member rows
 * are accumulated in Double and the mean is rounded to Single once: two
 * summation orders give the same Single unless the Double sums straddle a
 * rounding boundary of the Single (about 1e-9 per coordinate), which is why the
 * split over GPUs (gsc_split_*) reproduces the single-GPU centroids. */
int gsc_lloyd(gsc_ctx *ctx, const float *X, int N, int D, float *centroids,
              int K, int iters, int32_t *labels);

/* Oversized single frame (BASELINE.json configs[3], SURVEY.md 8e): the points of
 * ONE frame are split over several GPUs, one context per GPU holding a shard.
 * Per Lloyd iteration: gsc_split_step writes this shard's partial sums into
 * acc_dev, double[K][D+1] in DEVICE memory owned by the caller (D sums, then
 * the member count); the caller all-reduces acc_dev over the ranks (NCCL); then
 * gsc_split_update turns the reduced buffer into the new centroids (empty
 * clusters keep theirs).  Every call returns with the context stream idle; the
 * caller synchronises its own collective before gsc_split_update. */
int gsc_split_begin(gsc_ctx *ctx, const float *X, int N, int D,
                    const float *centroids, int K);
int gsc_split_step(gsc_ctx *ctx, double *acc_dev);
int gsc_split_update(gsc_ctx *ctx, const double *acc_dev);
/* final assignment against the last centroids; both outputs optional */
int gsc_split_end(gsc_ctx *ctx, float *centroids, int32_t *labels);

/* The same split with the collective INSIDE the library: NCCL (bound at run time from libnccl.so.2) over
 * NVLink / NVSwitch, one context per rank.  Rank 0 makes an id (gsc_split_unique_id) and hands the 128 bytes to
 * the other ranks by whatever transport the host has; every rank calls gsc_split_comm_init.  gsc_split_seed gives
 * all ranks the same start (yakmo's k-means++ on the first <= 524,288 rows of rank 0's shard, broadcast); gsc_split_lloyd runs
 * `iters` x (assign, Double partial sums, ncclAllReduce(sum) of K x (D+1) doubles, means) + a final assignment on
 * the context's stream without a host synchronisation inside the loop.  centroids: in = the start (identical on
 * every rank), out = the result (identical on every rank, and bit-identical to gsc_lloyd on the whole frame:
 * Double accumulation, one rounding to Single).  ms_out (optional): 3 doubles from CUDA events -- the loop, the
 * time inside the all-reduces, the first iteration.  Without gsc_split_comm_init the call runs on one rank. */
#define GSC_SPLIT_ID_BYTES 128
int gsc_split_unique_id(char *id /* [GSC_SPLIT_ID_BYTES] */);
int gsc_split_comm_init(gsc_ctx *ctx, int nranks, int rank, const char *id);
int gsc_split_comm_destroy(gsc_ctx *ctx);
int gsc_split_seed(gsc_ctx *ctx, const float *X_shard, int N, int D, int K, float *centroids);
int gsc_split_lloyd(gsc_ctx *ctx, const float *X_shard, int N, int D, float *centroids, int K, int iters,
                    int32_t *labels, double *ms_out);

/* Exact nearest centroid per row (ANN-style distance). dist optional. */
int gsc_assign(gsc_ctx *ctx, const float *X, int N, int D,
               const float *centroids, int K, int32_t *labels, float *dist);

/* enc:843-889: class means in the sample domain, population sort (FreePascal
 * quicksort order), dictionary quantisation.  means float[K][cs] and
 * counts/order int32[K] in dictionary order (order[i] = cluster of entry i),
 * dict int16[K][cs], datten/dattr uint8[K], entry int32[N] (dictionary entry
 * of every chunk's cluster); any output may be NULL. */
int gsc_build_dictionary(gsc_ctx *ctx, const int32_t *labels, const int16_t *pcm,
                         int64_t stride, int C, int S, const uint8_t *attr,
                         int cs, int K, int bits, int divider, float *means,
                         int32_t *order, int32_t *counts, int16_t *dict,
                         uint8_t *datten, uint8_t *dattr, int32_t *entry);

/* enc:915-965 KNNFit.  best int32[N] (variant row), use int32[R],
 * band (optional) int32[N] = rows inside the epsilon band. */
int gsc_knnfit(gsc_ctx *ctx, const int16_t *dict, const uint8_t *datten, int R,
               int cs, int bits, int divider, const int16_t *pcm,
               int64_t stride, int C, int S, int32_t *best, int32_t *use,
               int32_t *band);

/* kmeans_mode 3: enc:915-965 the way the binary runs it -- an ANN kd-tree over the 4R variant rows, the 64 nearest
 * rows per chunk (standard search, ties in visit order), the lowest row index within epsilon of the nearest.
 * Bit-identical to the oracle's kd-tree KNNFit.  best int32[N] (variant row), use int32[R]. */
int gsc_knnfit_kdtree(gsc_ctx *ctx, const int16_t *dict, const uint8_t *datten, int R, int cs, int bits, int divider,
                      const int16_t *pcm, int64_t stride, int C, int S, int32_t *best, int32_t *use);

/* enc:970-977: prune unused entries, sort by use count (FreePascal quicksort
 * order), renumber.  remap int32[R] old->new or -1; order int32[R]. */
int gsc_finalize_dictionary(gsc_ctx *ctx, const int32_t *use, int R,
                            int32_t *remap, int32_t *order, int *new_R);

/* ===================================================================== */
/* 3. Whole frames (enc:1433-1447 DoFrame), batched                       */
/* ===================================================================== */

typedef struct gsc_params {
    int32_t chunk_size;        /* -cs   enc:1496 (4)    */
    int32_t chunk_bit_depth;   /* -cbd  enc:1495 (8|12) */
    int32_t chunks_per_frame;  /* -cpf  enc:1505 (<=4096) */
    int32_t precision;         /* -pr   enc:1503 (3); 0 = passthrough */
    int32_t max_passes;        /* CMaxIterations enc:703 (100) */
    int32_t kmeans_mode;       /* 0 online (reference rule, exact search), 1 Lloyd,
                                  3 online through the reference's ANN kd-tree searches (k-means and KNNFit;
                                  chunk sizes 2 and 4) */
    int32_t lloyd_iters;       /* mode 1 */
    int32_t reserved;
} gsc_params;

void gsc_default_params(gsc_params *p);

typedef struct gsc_frame_desc {
    const int16_t *pcm;        /* planar [C][>=S], first sample of the frame */
    int64_t stride;            /* samples between channel rows */
    int32_t channels;
    int32_t samples;           /* per channel, > 0 */
} gsc_frame_desc;

typedef struct gsc_frame_result {
    /* caller-allocated */
    int16_t *dict;             /* [chunks_per_frame or N][cs] capacity */
    uint8_t *datten;           /* [same capacity] */
    int32_t *index;            /* [N] final dictionary index per chunk */
    uint8_t *attr;             /* [N] bit1 Negative, bit0 Reversed */
    /* written by the library */
    int32_t N, R, divider, passes;
    double  err;               /* last KNNScanReduce residual (enc:764) */
    int32_t overfull;          /* queries with > 64 rows in the epsilon band */
    int32_t reserved;
} gsc_frame_result;

/* Capacity (entries) the caller must provide for dict/datten of a frame. */
int gsc_dict_capacity(const gsc_params *p, int channels, int samples);

/* results may be NULL when only the packed stream / quality are wanted
 * (gsc_fetch_stream, gsc_fetch_quality): nothing but those is copied back. */
int gsc_encode_frames(gsc_ctx *ctx, const gsc_frame_desc *frames, int n_frames,
                      const gsc_params *params, gsc_frame_result *results);

/* Same pipeline with the PCM of all frames already resident on the device
 * (used by bench.py's device-resident `value` leg): `pcm_dev` is one device
 * buffer, frames[i].pcm are DEVICE pointers into it.  Results stay on the
 * device until gsc_fetch_results. */
int gsc_encode_frames_dev(gsc_ctx *ctx, const gsc_frame_desc *frames_devptr,
                          int n_frames, const gsc_params *params);
int gsc_fetch_results(gsc_ctx *ctx, int n_frames, gsc_frame_result *results);

/* SURVEY.md 8(f3): the .gsc bytes (TFrame.SaveStream, enc:980-1107) of the last gsc_encode_frames* batch, packed
 * on the device: header, attenuation nibbles, 8/12-bit dictionary samples, variable-length index codes.  The
 * frames' streams are written to `out` back to back in frame order (enc:1208-1214); frame_bytes[n_frames] and
 * *total are optional.  out = NULL only sizes.  sample_rate goes into the frame header (enc:994). */
int gsc_fetch_stream(gsc_ctx *ctx, int n_frames, int sample_rate, uint8_t *out, int64_t cap,
                     int64_t *frame_bytes, int64_t *total);
/* SURVEY.md 8(f2): encoder-side reconstruction (enc:487-522, 1518-1582) of the last batch compared with its PCM:
 * sq_err[i] = sum over frame i of (src - dst)^2 in int16 units (exact), samples[i] = its sample count.
 * PsyADelta (enc:1862-1880) = sqrt(sum sq_err / sum samples).  The PCM of the batch must still be on the
 * device (always true after gsc_encode_frames; after gsc_encode_frames_dev while the caller keeps its buffer). */
int gsc_fetch_quality(gsc_ctx *ctx, int n_frames, uint64_t *sq_err, int64_t *samples);

/* Cross-check paths for the parity tests, per context (results are identical by construction; the tests check
 * that).  flags = OR of: */
#define GSC_DBG_ONLINE_EXACT  1u   /* online k-means scores every centroid exactly instead of using its filter */
#define GSC_DBG_SEED_FULLSCAN 2u   /* seeding with the round-1 kernel: every step scans all points (block scan) */
#define GSC_DBG_SEED_SERIAL   4u   /* ... and evaluates yakmo's float prefix sum with a one-warp serial chain */
#define GSC_DBG_KNNFIT_DENSE  8u   /* KNNFit scans all entries twice instead of walking the norm window */
#define GSC_DBG_LLOYD_OWNER   16u  /* Lloyd update by per-cluster owner threads (ordered sums) instead of the scatter */
#define GSC_DBG_ONLINE_BATCHED 32u /* K <= 256: the batched CTA-per-frame kernel instead of the warp-per-frame one */
#define GSC_DBG_LABEL_SCAN     64u /* per-cluster sums by scanning all labels per cluster (O(K*N)) instead of member lists */
#define GSC_DBG_DIVIDER_V1     128u /* FindAttenuationDivider with the per-thread loop that divides in the inner loop */
#define GSC_DBG_KDTREE_SERIAL  256u /* kmeans_mode 3: the kd-tree k-means searches one point per round (no speculation) */
int gsc_ctx_set_debug(gsc_ctx *ctx, unsigned flags);
/* Exhaustive self-check of the tabulated-reciprocal division used by the attenuation-divider kernel at `bits`. */
int gsc_selftest_divider_division(gsc_ctx *ctx, int bits, uint64_t *mismatches);
/* Debug: counters of the last online k-means launch, 16 x uint64 per frame:
 * batches, points, re-filtered points, resolver rounds, full candidate lists,
 * candidates (lane 0), commits of a centroid already moved in the same batch; slots 8..15
 * are zero except in debug builds (GSC_ONLINE_CHECKS, GSC_ONLINE_TIMING).  After a kmeans_mode 3 k-means (all passes):
 * speculation rounds, points committed, lane searches, visit lists that overflowed. */
int gsc_debug_online_counters(gsc_ctx *ctx, unsigned long long *out, int n_frames);
/* Debug: counters of the last seeding launch, 8 x uint64 per frame: cycles of seed pick, distance pass,
 * summaries + chain, number of steps; windows evaluated exactly, blocks visited, windows re-summarised, chain cycles. */
int gsc_debug_seed_counters(gsc_ctx *ctx, unsigned long long *out, int n_frames);

/* SURVEY.md 8(f1): the frame planner's power scan and boundary selection (TEncoder.PrepareFrames enc:1374-1425, with
 * the int16 -> Double staging of enc:1282-1285) on the device.  pcm planar [C][S], S already padded to the block size
 * (enc:1319-1323); block = ChunkSize (under-sampling 1, blend 0).  starts[0..*n_frames) = first sample of every frame,
 * exactly what the reference's sequential Double sums give (the sums are evaluated bit-exactly in parallel, see
 * csrc/gsc_plan.cuh).  stats (optional, 4 values): windows added element by element in pass 1 / pass 2, boundary
 * iterations (1 = every candidate was right), windows of pass 1. */
int gsc_plan_frames(gsc_ctx *ctx, const int16_t *pcm, int64_t stride, int C, int64_t S, int sample_rate,
                    double frame_length_ms, double vfr, int block, int64_t *starts, int max_frames, int *n_frames,
                    uint64_t *stats);
int gsc_plan_frames_dev(gsc_ctx *ctx, const int16_t *pcm_dev, int64_t stride, int C, int64_t S, int sample_rate,
                        double frame_length_ms, double vfr, int block, int64_t *starts, int max_frames, int *n_frames,
                        uint64_t *stats);

/* The library's natural logarithm (csrc/gsc_log.h: correctly rounded, plain IEEE double operations; the cepstral
 * features enc:316-318 go through it) over a host array, so that a host can compare it value by value. */
int gsc_log_array(gsc_ctx *ctx, const double *x, int64_t n, double *y);

/* FP32 FFMA throughput probe (roofline denominator for the k-means / search
 * kernels): returns measured TFLOP/s on the context's device. */
int gsc_fp32_peak_probe(gsc_ctx *ctx, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* GSC_CUDA_H */
