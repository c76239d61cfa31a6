/*
 * gsc_host.h -- C ABI of libgsc_host.so: the host side of the SoundChunks
 * encoder around libgsc_cuda.so (include/gsc_cuda.h).
 *
 * The reference's host is one FreePascal program (encoder/encoder.lpr); its
 * toolchain (fpc/lazbuild) is absent here, so the host steps that stay on the
 * CPU are restated in C++ with the reference's option names, defaults and
 * error behaviour.  enc:L = /root/reference/encoder/encoder.lpr line L,
 * dec:L = /root/reference/decoder/decoder.lpr line L.
 *
 *   TEncoder.Load            enc:1111-1152   gsch_load_wav
 *   TEncoder.PrepareFrames   enc:1294-1429   gsch_plan_frames
 *   TEncoder.MakeFrames      enc:1431-1451   gsch_encode_pcm  (frames sharded over GPUs,
 *                                             one host thread + one gsc_ctx per device,
 *                                             DoFrame itself runs in libgsc_cuda.so)
 *   TFrame.SaveStream        enc:980-1107    gsch_write_frame
 *   TEncoder.SaveGSC         enc:1181-1215   gsch_encode_file
 *   TEncoder.MakeDstData +   enc:487-522,    gsch_reconstruct_frame, gsch_psy_a_delta
 *     ComputePsyADelta       1518-1582, 1862-1880
 *   GSCUnpack                dec:37-220      gsch_decode, gsch_decode_file
 *   option parsing           enc:201-227, 1985-1998   gsch_parse_option
 *
 * Nothing here computes the hot path: without a usable sm_100 device
 * gsch_encode_* fail with the error text of libgsc_cuda.so.
 */
#ifndef GSC_HOST_H
#define GSC_HOST_H

#include <stdint.h>
#include "gsc_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gsch_options {
    int32_t bitrate;            /* -br   kbit/s, -1 = unlimited        enc:1491 */
    int32_t precision;          /* -pr   enc:1503 (3)                           */
    double  low_cut;            /* -lc   enc:1493 (0)     must stay 0           */
    double  high_cut;           /* -hc   enc:1494 (24000) must stay >= sr/2     */
    double  vfr;                /* -vfr  enc:1499 (1.0)                         */
    double  frame_length_ms;    /* -fl   enc:1501 (4000)                        */
    int32_t chunk_bit_depth;    /* -cbd  enc:1495 (8)                           */
    int32_t chunk_size;         /* -cs   enc:1496 (4)                           */
    int32_t chunks_per_frame;   /* -cpf  enc:1505 (4096), clamped 256..4096     */
    int32_t chunk_blend;        /* -cb   enc:1500 (0)     must stay 0           */
    int32_t verbose;            /* -v                                           */
    /* not in the reference CLI */
    int32_t kmeans_mode;        /* 0 online rule (reference), 1 batch Lloyd (-lloyd),
                                   3 reference's kd-tree searches (-kdtree)     */
    int32_t lloyd_iters;
    int32_t max_passes;         /* CMaxIterations enc:703 (100)                 */
    int32_t devices;            /* GPUs to shard frames over, 0 = all visible   */
    int32_t frames_per_call;    /* frames per gsc_encode_frames call and device */
} gsch_options;

typedef struct gsch_report {
    int32_t frames, channels, sample_rate, chunks_per_frame, devices;
    int64_t samples;            /* per channel, after padding (enc:1319)        */
    int64_t gsc_bytes;
    double  bitrate_kbps;       /* enc:1199                                     */
    double  psy_a_delta;        /* enc:2026-2027                                */
    double  encode_seconds;     /* MakeFrames wall time                         */
    int64_t overfull;           /* queries with > 64 rows in the epsilon band   */
} gsch_report;

const char *gsch_last_error(void);
void gsch_default_options(gsch_options *o);
/* One command-line argument in the reference's `-xx<value>` form (enc:1985-1998).
 * Returns 0 if recognised, 1 if not an option of this encoder. */
int gsch_parse_option(gsch_options *o, const char *arg);

/* enc:1111-1152.  Reads a 16-bit PCM WAV with the reference's fixed 44-byte
 * header assumption; *pcm is planar [C][S], caller frees with gsch_free. */
int gsch_load_wav(const char *path, int16_t **pcm, int *channels, int64_t *samples, int *sample_rate);
int gsch_save_wav(const char *path, const int16_t *pcm_planar, int channels, int64_t samples, int sample_rate);
void gsch_free(void *p);

/* enc:1319: sample count rounded up to a whole block. */
int64_t gsch_padded_samples(int64_t samples, const gsch_options *o);
/* enc:1337-1351: solve ChunksPerFrame from -br (o->chunks_per_frame in/out),
 * enc:1374-1425: power-driven frame cut.  pcm planar, already padded.
 * Returns the number of frames (starts[k] = first sample of frame k). */
int gsch_plan_frames(const int16_t *pcm, int64_t stride, int channels, int64_t samples, int sample_rate,
                     gsch_options *o, int64_t *starts, int max_frames);

/* enc:980-1107 for one frame; buf may be NULL to size.  Returns bytes. */
int64_t gsch_write_frame(const gsc_frame_result *f, int channels, int cs, int bits, int sample_rate,
                         uint8_t *buf, int64_t cap);
/* dec:37-220.  out planar [C][cap_samples] with row stride cap_samples; may be
 * NULL to size.  Returns samples per channel, -1 on a malformed stream. */
int64_t gsch_decode(const uint8_t *gsc, int64_t len, int16_t *out, int64_t cap_samples, int *channels,
                    int *sample_rate);
/* enc:487-522 + 1518-1582 for one frame into planar out (row stride `stride`). */
void gsch_reconstruct_frame(const gsc_frame_result *f, int channels, int samples, int cs, int bits,
                            int16_t *out, int64_t stride);
/* enc:1862-1880 */
double gsch_psy_a_delta(const int16_t *a, const int16_t *b, int64_t n);

/* Load .. SaveGSC on PCM in memory (enc:2016-2024).  *gsc is malloc'ed. */
int gsch_encode_pcm(const int16_t *pcm, int64_t stride, int channels, int64_t samples, int sample_rate,
                    const gsch_options *o, uint8_t **gsc, int64_t *gsc_len, gsch_report *rep);
int gsch_encode_file(const char *wav_path, const char *gsc_path, const gsch_options *o, gsch_report *rep);
int gsch_decode_file(const char *gsc_path, const char *wav_path);

#ifdef __cplusplus
}
#endif
#endif /* GSC_HOST_H */
