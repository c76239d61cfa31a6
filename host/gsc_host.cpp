// gsc_host.cpp -- libgsc_host.so: the CPU-resident steps of the SoundChunks encoder
// around libgsc_cuda.so (include/gsc_host.h).  C++17, no CUDA.
//
// What stays on the host in the reference stays on the host here: WAV I/O,
// frame planning, the .gsc bitstream writer, the quality print.  DoFrame
// (enc:1433-1447) is NOT here: MakeFrames hands whole frames to
// gsc_encode_frames, sharded over the visible GPUs.
#include "../include/gsc_host.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string t_err;

int fail(const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_err = buf;
    return 1;
}

inline double float_sample(int16_t s) { return (double)s / 32767.0; }   // enc:1643-1646

inline int16_t make16(double smp) {                                      // enc:1638-1641
    double r = std::nearbyint(smp * 32767.0);
    if (r < -32768.0) r = -32768.0;
    if (r > 32767.0) r = 32767.0;
    return (int16_t)r;
}

inline double dequant(int16_t q, int bits, int atten, bool neg, double law) {   // enc:1665-1680
    double coeff = 1.0;
    for (int i = 0; i <= atten; ++i) coeff += (double)i * law;
    const double obd = (double)((1 << (bits - 1)) - 1);
    int16_t s = q;
    if (neg) s = (int16_t)(-s);
    double r = (double)s / (obd * coeff);
    return std::min(1.0, std::max(-1.0, r));
}

// little-endian byte sink that can also just count
struct Sink {
    uint8_t *buf;
    int64_t cap, pos = 0;
    Sink(uint8_t *b, int64_t c) : buf(b), cap(c) {}
    void u8(unsigned v) { if (buf && pos < cap) buf[pos] = (uint8_t)v; ++pos; }
    void u16(unsigned v) { u8(v & 0xff); u8((v >> 8) & 0xff); }
    void u32(uint32_t v) { u16(v & 0xffff); u16(v >> 16); }
};

inline int bit_scan_reverse(unsigned v) { int r = 0; while (v >>= 1) ++r; return r; }
// enc:1054-1060: number of extra 3-bit groups of an index
inline int index_groups(int index) { return index == 0 ? 0 : bit_scan_reverse((unsigned)index) / 3; }

bool starts_with(const char *s, const char *p) { return strncmp(s, p, strlen(p)) == 0; }

double param_value(const char *arg, const char *name, double def) {   // enc:219-227 StrToFloatDef
    const char *v = arg + strlen(name);
    if (!*v) return def;
    char *end = nullptr;
    double x = strtod(v, &end);
    return (end && *end == 0) ? x : def;
}

template <class T> T clampv(T v, T lo, T hi) { return v < lo ? lo : (v > hi ? hi : v); }
long pascal_round(double v) { return (long)std::nearbyint(v); }   // FreePascal round = half to even

}  // namespace

extern "C" const char *gsch_last_error(void) { return t_err.c_str(); }

extern "C" void gsch_default_options(gsch_options *o) {
    o->bitrate = -1;            // enc:1491
    o->precision = 3;           // enc:1503
    o->low_cut = 0.0;           // enc:1493
    o->high_cut = 24000.0;      // enc:1494
    o->vfr = 1.0;               // enc:1499
    o->frame_length_ms = 4000;  // enc:1501
    o->chunk_bit_depth = 8;     // enc:1495
    o->chunk_size = 4;          // enc:1496
    o->chunks_per_frame = 4096; // enc:1505
    o->chunk_blend = 0;         // enc:1500
    o->verbose = 0;
    o->kmeans_mode = 0;
    o->lloyd_iters = 30;
    o->max_passes = 100;        // enc:703
    o->devices = 0;
    o->frames_per_call = 592;
}

extern "C" int gsch_parse_option(gsch_options *o, const char *a) {
    // prefixes are tested longest first: the reference's AnsiStartsStr would let "-c" style
    // prefixes shadow each other, its option names do not collide except -cb / -cbd (enc:1995)
    if (!a || a[0] != '-') return 1;
    if (starts_with(a, "-br")) { o->bitrate = (int)pascal_round(param_value(a, "-br", o->bitrate)); return 0; }
    if (starts_with(a, "-pr")) { o->precision = (int)pascal_round(param_value(a, "-pr", o->precision)); return 0; }
    if (starts_with(a, "-lc")) { o->low_cut = param_value(a, "-lc", o->low_cut); return 0; }
    if (starts_with(a, "-hc")) { o->high_cut = param_value(a, "-hc", o->high_cut); return 0; }
    if (starts_with(a, "-vfr")) { o->vfr = clampv(param_value(a, "-vfr", o->vfr), 0.0, 1.0); return 0; }
    if (starts_with(a, "-fl")) { o->frame_length_ms = std::max(param_value(a, "-fl", o->frame_length_ms), 1.0); return 0; }
    if (starts_with(a, "-cbd")) { o->chunk_bit_depth = clampv((int)pascal_round(param_value(a, "-cbd", o->chunk_bit_depth)), 1, 16); return 0; }
    if (starts_with(a, "-cs")) { o->chunk_size = (int)pascal_round(param_value(a, "-cs", o->chunk_size)); return 0; }
    if (starts_with(a, "-cpf")) { o->chunks_per_frame = clampv((int)pascal_round(param_value(a, "-cpf", o->chunks_per_frame)), 256, 4096); return 0; }
    if (starts_with(a, "-cb")) { o->chunk_blend = (int)pascal_round(param_value(a, "-cb", o->chunk_blend)); return 0; }
    if (strcmp(a, "-v") == 0) { o->verbose = 1; return 0; }
    // extensions
    if (starts_with(a, "-lloyd")) { o->kmeans_mode = 1; o->lloyd_iters = (int)param_value(a, "-lloyd", o->lloyd_iters); return 0; }
    if (strcmp(a, "-kdtree") == 0) { o->kmeans_mode = 3; return 0; }
    if (starts_with(a, "-gpus")) { o->devices = (int)param_value(a, "-gpus", o->devices); return 0; }
    return 1;
}

// ---------------------------------------------------------------------------------------------
// WAV (enc:1111-1152, 1154-1179; extern.pas:24-47 TWavHeader)
// ---------------------------------------------------------------------------------------------
extern "C" int gsch_load_wav(const char *path, int16_t **pcm, int *channels, int64_t *samples, int *sample_rate) {
    FILE *f = fopen(path, "rb");
    if (!f) return fail("cannot open %s", path);
    uint8_t hdr[44];
    if (fread(hdr, 1, 44, f) != 44) { fclose(f); return fail("%s: short WAV header", path); }
    int32_t sr; uint16_t ch;
    memcpy(&sr, hdr + 0x18, 4);   // enc:1134
    memcpy(&ch, hdr + 0x16, 2);   // enc:1135
    if (ch == 0 || sr <= 0) { fclose(f); return fail("%s: bad WAV header", path); }
    fseek(f, 0, SEEK_END);
    long size = ftell(f);
    fseek(f, 44, SEEK_SET);
    const int64_t S = (size - 44) / (2 * (int64_t)ch);   // enc:1137
    std::vector<int16_t> inter((size_t)S * ch);
    if (S > 0 && fread(inter.data(), 2, (size_t)S * ch, f) != (size_t)S * ch) { fclose(f); return fail("%s: short read", path); }
    fclose(f);
    int16_t *out = (int16_t *)malloc(sizeof(int16_t) * (size_t)std::max<int64_t>(S, 1) * ch);
    if (!out) return fail("out of memory");
    for (int64_t i = 0; i < S; ++i)
        for (int j = 0; j < ch; ++j) out[(size_t)j * S + i] = inter[(size_t)i * ch + j];   // enc:1143-1145
    *pcm = out; *channels = ch; *samples = S; *sample_rate = sr;
    return 0;
}

extern "C" int gsch_save_wav(const char *path, const int16_t *pcm, int channels, int64_t samples, int sample_rate) {
    FILE *f = fopen(path, "wb");
    if (!f) return fail("cannot create %s", path);
    const uint32_t data = (uint32_t)(samples * channels * 2);
    uint8_t h[44];
    auto p32 = [&](int o, uint32_t v) { memcpy(h + o, &v, 4); };
    auto p16 = [&](int o, uint16_t v) { memcpy(h + o, &v, 2); };
    memcpy(h, "RIFF", 4); p32(4, 36 + data); memcpy(h + 8, "WAVEfmt ", 8); p32(16, 16); p16(20, 1);
    p16(22, (uint16_t)channels); p32(24, (uint32_t)sample_rate); p32(28, (uint32_t)(sample_rate * channels * 2));
    p16(32, (uint16_t)(channels * 2)); p16(34, 16); memcpy(h + 36, "data", 4); p32(40, data);
    fwrite(h, 1, 44, f);
    std::vector<int16_t> inter((size_t)samples * channels);
    for (int64_t i = 0; i < samples; ++i)
        for (int j = 0; j < channels; ++j) inter[(size_t)i * channels + j] = pcm[(size_t)j * samples + i];
    fwrite(inter.data(), 2, inter.size(), f);
    fclose(f);
    return 0;
}

extern "C" void gsch_free(void *p) { free(p); }

// ---------------------------------------------------------------------------------------------
// PrepareFrames (enc:1294-1429)
// ---------------------------------------------------------------------------------------------
static int check_options(const gsch_options *o, int sample_rate) {
    if (!o) return fail("null options");
    if (o->chunk_blend != 0) return fail("-cb: chunk blend is not supported (decoder.lpr asserts ChunkBlend = 0, dec:108)");
    if (o->chunk_size != 2 && o->chunk_size != 4 && o->chunk_size != 8) return fail("-cs%d: chunk size must be 2, 4 or 8", o->chunk_size);
    if (o->chunk_bit_depth != 8 && o->chunk_bit_depth != 12) return fail("-cbd%d: chunk bit depth must be 8 or 12 (enc:1041)", o->chunk_bit_depth);
    if (o->low_cut != 0.0 || (sample_rate > 0 && o->high_cut < sample_rate / 2.0))
        return fail("-lc/-hc: the band-pass pre-filter (enc:1466-1484) is outside the hot path and not provided");
    return 0;
}

extern "C" int64_t gsch_padded_samples(int64_t S, const gsch_options *o) {
    const int64_t block = o->chunk_size - o->chunk_blend;   // underSample = 1 at the default cut-offs, enc:1312-1315
    return S <= 0 ? 0 : ((S - 1) / block + 1) * block;      // enc:1319
}

// enc:1325-1351: largest ChunksPerFrame whose projected size fits the bit rate (host scalar logic)
static int solve_chunks_per_frame(gsch_options *o, int C, int64_t S, int sample_rate, int frameCount) {
    const int block = o->chunk_size - o->chunk_blend;
    {
        const double projected = o->bitrate > 0 ? std::ceil(((double)S / sample_rate) * ((double)o->bitrate * 1024.0 / 8.0)) : 2147483647.0;
        int cpf = o->chunks_per_frame + 1;
        double tentative;
        do {
            --cpf;
            const double bandCost = ((double)S * C * (std::log2((double)cpf) + (1 + 2) + 1 + 1)) / (8.0 * block * 1);
            const double frameCost = ((double)cpf * o->chunk_size) * o->chunk_bit_depth / 8.0 + (double)cpf * 4 / 8.0 + (4 * 2 + 4 + 1 * 4);
            tentative = std::nearbyint(0.0 + bandCost * 0.8 + frameCount * frameCost);
        } while (!(tentative <= projected || cpf <= 1));
        o->chunks_per_frame = cpf;
        if (cpf <= 0) { fail("Null ChunksPerFrame! (BitRate too low)"); return -1; }   // enc:1360
    }
    return 0;
}

extern "C" int gsch_plan_frames(const int16_t *pcm, int64_t stride, int C, int64_t S, int sample_rate, gsch_options *o,
                                int64_t *starts, int max_frames) {
    if (!pcm || C <= 0 || S <= 0 || sample_rate <= 0 || !starts || max_frames <= 0) { fail("gsch_plan_frames: bad arguments"); return -1; }
    if (check_options(o, sample_rate)) return -1;
    const int block = o->chunk_size - o->chunk_blend;
    const int frameCount = (int)std::ceil((double)S / ((double)sample_rate * (o->frame_length_ms / 1000.0)));   // enc:1335
    if (solve_chunks_per_frame(o, C, S, sample_rate, frameCount)) return -1;
    auto rms_at = [&](int64_t i) {
        double smp = 0.0;
        for (int j = 0; j < C; ++j) { const double x = float_sample(pcm[(size_t)j * stride + i]); smp += x * x; }
        return std::sqrt(smp / (double)C);
    };
    double avg = 0.0;   // enc:1376-1380
    for (int j = 0; j < C; ++j)
        for (int64_t i = 0; i < S; ++i) { const double x = float_sample(pcm[(size_t)j * stride + i]); avg += x * x; }
    avg = std::sqrt(avg / ((double)S * (double)C));
    std::vector<double> w((size_t)S);
    double total = 0.0;   // enc:1382-1391
    for (int64_t i = 0; i < S; ++i) { w[i] = 1.0 - (avg + (rms_at(i) - avg) * o->vfr); total += w[i]; }
    const double per = total / (double)frameCount;   // enc:1393
    int k = 0;
    int64_t next = 0;
    double cur = 0.0;
    for (int64_t i = 0; i < S; ++i) {   // enc:1401-1420
        cur += w[i];
        if (i % block == 0 && cur >= per) {
            if (k < max_frames) starts[k] = next;
            cur = 0.0; next = i; ++k;
        }
    }
    if (k < max_frames) starts[k] = next;   // enc:1422-1423
    ++k;
    if (k > max_frames) { fail("gsch_plan_frames: %d frames, room for %d", k, max_frames); return -1; }
    return k;
}

// ---------------------------------------------------------------------------------------------
// TFrame.SaveStream (enc:980-1107)
// ---------------------------------------------------------------------------------------------
extern "C" int64_t gsch_write_frame(const gsc_frame_result *f, int C, int cs, int bits, int sample_rate, uint8_t *buf,
                                    int64_t cap) {
    Sink w(buf, cap);
    w.u16(((unsigned)C << 8) | 1u);                 // StreamVersion = 1, ChannelCount   enc:988-989
    w.u16((unsigned)f->R);                          // ChunkCount | (BandCount-1) << 13  enc:990-991
    w.u16(((unsigned)cs << 8) | (unsigned)bits);    // enc:992-993
    w.u32((uint32_t)sample_rate);                   // | ChunkBlend << 24                enc:994-995
    w.u16((unsigned)f->divider);                    // enc:996-997
    for (int j = 0; j + 1 < f->R; j += 2) w.u8(((unsigned)f->datten[j] << 4) | f->datten[j + 1]);   // enc:1003-1008
    if (f->R & 1) w.u8((unsigned)f->datten[f->R - 1] << 4);                                        // enc:1009-1011
    if (bits == 8) {                                // enc:1015-1018
        for (int j = 0; j < f->R * cs; ++j) w.u8((unsigned)(f->dict[j] + 128) & 0xff);
    } else {                                        // 12-bit pairs in 3 bytes, enc:1019-1039
        for (int j = 0; j < f->R; ++j) {
            const int16_t *d = f->dict + (size_t)j * cs;
            for (int k = 0; k + 1 < cs; k += 2) {
                const int s1 = d[k] + 2048, s2 = d[k + 1] + 2048;
                w.u8(((s1 >> 4) & 0xf0) | ((s2 >> 8) & 0x0f));
                w.u8(s1 & 0xff);
                w.u8(s2 & 0xff);
            }
            if (cs & 1) { const int s1 = d[cs - 1] + 2048; w.u8((s1 >> 4) & 0xf0); w.u8(s1 & 0xff); }
        }
    }
    w.u32((uint32_t)(f->N / C));                    // FrameLength: indexes per channel  enc:1048
    uint32_t acc = 0;
    int nbits = 0, prevGroups = -1;
    for (int j = 0; j < f->N; ++j) {                // enc:1052-1098, LSB first, flushed in 16-bit words
        const int idx = f->index[j];
        const int groups = index_groups(idx);
        uint32_t code = 0;
        int sz = 0;
        code |= (uint32_t)((f->attr[j] >> 1) & 1) << sz++;   // Negative
        code |= (uint32_t)(f->attr[j] & 1) << sz++;          // Reversed
        if (groups == prevGroups) { ++sz; }                  // NewHeader = 0
        else { code |= 1u << sz++; code |= (uint32_t)groups << sz; sz += 2; }
        for (int k = groups; k >= 0; --k) { code |= (uint32_t)((idx >> (3 * k)) & 7) << sz; sz += 3; }
        prevGroups = groups;
        acc |= code << nbits;
        nbits += sz;
        if (nbits >= 16) { w.u16(acc & 0xffff); acc >>= 16; nbits -= 16; }
    }
    if (nbits > 0) w.u16(acc & 0xffff);             // enc:1100-1105
    return w.pos;
}

// ---------------------------------------------------------------------------------------------
// GSCUnpack (dec:37-220)
// ---------------------------------------------------------------------------------------------
namespace {
struct BitReader {
    const uint8_t *g; int64_t len; int64_t &pos; uint32_t acc = 0; int cnt = 0;
    BitReader(const uint8_t *g_, int64_t l, int64_t &p) : g(g_), len(l), pos(p) {}
    void fill() {   // dec:44-56
        if (cnt < 16 && pos < len) {
            uint32_t w = g[pos] | ((pos + 1 < len) ? ((uint32_t)g[pos + 1] << 8) : 0u);
            pos += 2; acc |= w << cnt; cnt += 16;
        }
    }
    int get(int n) { int v = (int)(acc & ((1u << n) - 1)); acc >>= n; cnt -= n; return v; }
};
}  // namespace

extern "C" int64_t gsch_decode(const uint8_t *g, int64_t len, int16_t *out, int64_t cap, int *channels, int *sample_rate) {
    const int32_t attrMul = (int32_t)std::nearbyint(32768.0 * (32767.0 / 2047.0));   // CAttrMul dec:6
    int64_t pos = 0, written = 0;   // written = samples per channel so far
    int C = 0;
    while (pos != len) {
        if (pos + 14 > len) return -1;
        const int version = g[pos];                                   // dec:76
        C = g[pos + 1];
        const int R = (g[pos + 2] | (g[pos + 3] << 8)) & 0x1fff;      // dec:78-79
        const int bits = g[pos + 4], cs = g[pos + 5];
        uint32_t sr; memcpy(&sr, g + pos + 6, 4);
        const int blend = (int)(sr >> 24); sr &= 0xffffffu;
        const int divider = g[pos + 10] | (g[pos + 11] << 8);
        pos += 12;
        if (blend != 0 || cs <= 0 || cs > 64 || C <= 0 || C > 16 || divider <= 0) return -1;   // dec:108
        if (channels) *channels = C;
        if (sample_rate) *sample_rate = (int)sr;
        int32_t lut[2][16];                                            // dec:88-96
        double law = 1.0 / (double)divider, lawAcc = 1.0;
        for (int i = 0; i <= 15; ++i) {
            lawAcc += law * (double)i;
            lut[0][i] = (int32_t)std::nearbyint((double)attrMul / lawAcc);
            lut[1][i] = -lut[0][i];
        }
        std::vector<uint8_t> att((size_t)std::max(R, 1));
        std::vector<int16_t> ch((size_t)std::max(R, 1) * cs);
        if (pos + (R + 1) / 2 > len) return -1;
        for (int i = 0; i + 1 < R; i += 2) { const int b = g[pos++]; att[i] = (uint8_t)(b >> 4); att[i + 1] = (uint8_t)(b & 15); }   // dec:115-120
        if (R & 1) { const int b = g[pos++]; att[R - 1] = (uint8_t)(b >> 4); }
        if (bits == 8) {                                               // dec:131-137
            if (pos + (int64_t)R * cs > len) return -1;
            for (int i = 0; i < R * cs; ++i) { const int b = g[pos++]; ch[i] = (int16_t)(((b - 128) * 2047) / 127); }
        } else if (bits == 12) {                                       // dec:138-158
            if (pos + (int64_t)R * ((cs / 2) * 3 + (cs & 1) * 2) > len) return -1;
            for (int i = 0; i < R; ++i) {
                for (int j = 0; j + 1 < cs; j += 2) {
                    const int b = g[pos++];
                    const int s1 = g[pos++] | ((b & 0xf0) << 4);
                    const int s2 = g[pos++] | ((b & 0x0f) << 8);
                    ch[(size_t)i * cs + j] = (int16_t)(s1 - 2048);
                    ch[(size_t)i * cs + j + 1] = (int16_t)(s2 - 2048);
                }
                if (cs & 1) { const int b = g[pos++]; const int s1 = g[pos++] | ((b & 0xf0) << 4); ch[(size_t)i * cs + cs - 1] = (int16_t)(s1 - 2048); }
            }
        } else return -1;
        if (pos + 4 > len) return -1;
        uint32_t flen; memcpy(&flen, g + pos, 4); pos += 4;            // dec:164
        BitReader br(g, len, pos);
        int header = -1;
        int idx[16], ng[16], rv[16];
        for (uint32_t i = 0; i < flen; ++i) {
            for (int k = 0; k < C; ++k) {                              // dec:174-193
                br.fill();
                ng[k] = br.get(1);
                rv[k] = version > 0 ? br.get(1) : 0;
                if (br.get(1)) header = br.get(2);
                br.fill();
                int v = 0;
                for (int j = 0; j <= header; ++j) v = (v << 3) | br.get(3);
                if (v >= R) return -1;
                idx[k] = v;
            }
            for (int j = 0; j < cs; ++j)                               // dec:195-202
                for (int k = 0; k < C; ++k) {
                    const int32_t a = lut[ng[k]][att[idx[k]]];
                    const int32_t s = ch[(size_t)idx[k] * cs + (rv[k] ? cs - 1 - j : j)];
                    const int16_t o = (int16_t)(((uint32_t)(a * s) >> 15) & 0xffff);
                    const int64_t p = written + (int64_t)i * cs + j;
                    if (out && p < cap) out[(size_t)k * cap + p] = o;
                }
        }
        written += (int64_t)flen * cs;
        if (br.cnt >= 16) pos -= 2;                                     // dec:205-209
    }
    return written;
}

// ---------------------------------------------------------------------------------------------
// reconstruction and quality print (enc:487-522, 1518-1582, 1862-1880)
// ---------------------------------------------------------------------------------------------
extern "C" void gsch_reconstruct_frame(const gsc_frame_result *f, int C, int S, int cs, int bits, int16_t *out,
                                       int64_t stride) {
    const double law = 1.0 / (double)f->divider;   // enc:561-564
    const int cc = f->N / C;
    for (int i = 0; i < cc; ++i)
        for (int c = 0; c < C; ++c) {
            const int n = i * C + c, e = f->index[n];
            const bool ng = (f->attr[n] >> 1) & 1, rv = f->attr[n] & 1;
            for (int j = 0; j < cs; ++j) {
                const int p = i * cs + j;
                if (p >= S) continue;
                out[(size_t)c * stride + p] = make16(dequant(f->dict[(size_t)e * cs + (rv ? cs - 1 - j : j)], bits, f->datten[e], ng, law));
            }
        }
}

extern "C" double gsch_psy_a_delta(const int16_t *a, const int16_t *b, int64_t n) {
    double r = 0.0;   // enc:1869-1879: samples copied to Double arrays, then CompareEuclidean(Double) enc:1804-1815
    for (int64_t i = 0; i < n; ++i) { const double d = (double)a[i] - (double)b[i]; r += d * d; }
    return n > 0 ? std::sqrt(r / (double)n) : 0.0;
}

// ---------------------------------------------------------------------------------------------
// MakeFrames (enc:1431-1451): frames are independent; shard them over the GPUs
// ---------------------------------------------------------------------------------------------
namespace {
struct FrameBuf {
    std::vector<int16_t> dict;
    std::vector<uint8_t> datten, attr;
    std::vector<int32_t> index;
};
}  // namespace

extern "C" int gsch_encode_pcm(const int16_t *pcm_in, int64_t stride_in, int C, int64_t S0, int sample_rate,
                               const gsch_options *opt, uint8_t **gsc, int64_t *gsc_len, gsch_report *rep) {
    if (!pcm_in || C <= 0 || S0 <= 0 || !opt || !gsc || !gsc_len) return fail("gsch_encode_pcm: bad arguments");
    if (check_options(opt, sample_rate)) return 1;
    gsch_options o = *opt;
    const int cs = o.chunk_size, bits = o.chunk_bit_depth;
    // enc:1317-1323: pad with zeros to a whole block
    const int64_t S = gsch_padded_samples(S0, &o);
    std::vector<int16_t> pcm((size_t)C * S, 0);
    for (int j = 0; j < C; ++j) memcpy(&pcm[(size_t)j * S], pcm_in + (size_t)j * stride_in, sizeof(int16_t) * (size_t)S0);
    // PrepareFrames (enc:1294-1429): the ChunksPerFrame solver is host scalar logic; the power scan and the boundary
    // selection over all samples run on the device (gsc_plan_frames, bit-exact; gsch_plan_frames is the host form)
    const int frameCount = (int)std::ceil((double)S / ((double)sample_rate * (o.frame_length_ms / 1000.0)));   // enc:1335
    if (solve_chunks_per_frame(&o, C, S, sample_rate, frameCount)) return 1;
    std::vector<int64_t> starts((size_t)frameCount * 4 + 16);
    int F = 0;
    {
        gsc_ctx *pctx = gsc_create(0);
        if (!pctx) return fail("no usable sm_100 CUDA device: %s", gsc_last_error());
        const int rc = gsc_plan_frames(pctx, pcm.data(), S, C, S, sample_rate, o.frame_length_ms, o.vfr, cs - o.chunk_blend,
                                       starts.data(), (int)starts.size(), &F, nullptr);
        if (rc != GSC_OK) { fail("gsc_plan_frames: %s", gsc_last_error()); gsc_destroy(pctx); return 1; }
        gsc_destroy(pctx);
    }
    if (F <= 0) return 1;
    starts.resize(F);
    std::vector<int> fsamples(F);
    for (int k = 0; k < F; ++k) fsamples[k] = (int)((k + 1 < F ? starts[k + 1] : S) - starts[k]);

    gsc_params P;
    gsc_default_params(&P);
    P.chunk_size = cs; P.chunk_bit_depth = bits; P.chunks_per_frame = o.chunks_per_frame; P.precision = o.precision;
    P.max_passes = o.max_passes; P.kmeans_mode = o.kmeans_mode; P.lloyd_iters = o.lloyd_iters;

    int ndev = gsc_device_count();
    if (ndev <= 0) return fail("no usable sm_100 CUDA device: %s", gsc_last_error());
    if (o.devices > 0) ndev = std::min(ndev, o.devices);
    ndev = std::min(ndev, F);

    // result storage
    std::vector<FrameBuf> bufs(F);
    std::vector<gsc_frame_result> res(F);
    const int cap = gsc_dict_capacity(&P, C, 0);
    for (int k = 0; k < F; ++k) {
        const int N = ((fsamples[k] - 1) / cs + 1) * C;   // enc:455
        bufs[k].dict.assign((size_t)std::max(cap, N <= cap ? N : cap) * cs, 0);
        bufs[k].datten.assign((size_t)std::max(cap, 1), 0);
        bufs[k].index.assign((size_t)N, 0);
        bufs[k].attr.assign((size_t)N, 0);
        memset(&res[k], 0, sizeof(res[k]));
        res[k].dict = bufs[k].dict.data(); res[k].datten = bufs[k].datten.data();
        res[k].index = bufs[k].index.data(); res[k].attr = bufs[k].attr.data();
    }
    // greedy longest-first assignment of frames to devices (SURVEY.md 8e)
    std::vector<int> order(F);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return fsamples[a] > fsamples[b]; });
    std::vector<std::vector<int>> shard(ndev);
    std::vector<int64_t> load(ndev, 0);
    for (int k : order) {
        int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        shard[d].push_back(k);
        load[d] += fsamples[k];
    }
    std::vector<std::string> errs(ndev);
    const auto t0 = std::chrono::steady_clock::now();
    auto worker = [&](int d) {
        gsc_ctx *ctx = gsc_create(d);
        if (!ctx) { errs[d] = gsc_last_error(); return; }
        std::sort(shard[d].begin(), shard[d].end());
        const int per = std::max(1, o.frames_per_call);
        for (size_t b = 0; b < shard[d].size() && errs[d].empty(); b += per) {
            const int n = (int)std::min<size_t>(per, shard[d].size() - b);
            std::vector<gsc_frame_desc> desc(n);
            std::vector<gsc_frame_result> r(n);
            for (int i = 0; i < n; ++i) {
                const int k = shard[d][b + i];
                desc[i].pcm = pcm.data() + starts[k]; desc[i].stride = S; desc[i].channels = C; desc[i].samples = fsamples[k];
                r[i] = res[k];
            }
            if (gsc_encode_frames(ctx, desc.data(), n, &P, r.data()) != GSC_OK) { errs[d] = gsc_last_error(); break; }
            for (int i = 0; i < n; ++i) res[shard[d][b + i]] = r[i];
        }
        gsc_destroy(ctx);
    };
    std::vector<std::thread> th;
    for (int d = 0; d < ndev; ++d) th.emplace_back(worker, d);
    for (auto &t : th) t.join();
    for (int d = 0; d < ndev; ++d) if (!errs[d].empty()) return fail("device %d: %s", d, errs[d].c_str());
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();

    // SaveStream: frames in index order (enc:1208-1214)
    int64_t total = 0;
    std::vector<int64_t> sizes(F);
    for (int k = 0; k < F; ++k) { sizes[k] = gsch_write_frame(&res[k], C, cs, bits, sample_rate, nullptr, 0); total += sizes[k]; }
    uint8_t *blob = (uint8_t *)malloc((size_t)std::max<int64_t>(total, 1));
    if (!blob) return fail("out of memory");
    int64_t off = 0;
    for (int k = 0; k < F; ++k) { gsch_write_frame(&res[k], C, cs, bits, sample_rate, blob + off, sizes[k]); off += sizes[k]; }
    *gsc = blob; *gsc_len = total;
    if (rep) {
        std::vector<int16_t> dst((size_t)C * S, 0);
        int64_t overfull = 0;
        for (int k = 0; k < F; ++k) {
            gsch_reconstruct_frame(&res[k], C, fsamples[k], cs, bits, dst.data() + starts[k], S);
            overfull += res[k].overfull;
        }
        rep->frames = F; rep->channels = C; rep->sample_rate = sample_rate; rep->chunks_per_frame = o.chunks_per_frame;
        rep->devices = ndev; rep->samples = S; rep->gsc_bytes = total;
        rep->bitrate_kbps = (double)total * (8.0 / 1024.0) / ((double)S / sample_rate);   // enc:1199
        rep->psy_a_delta = gsch_psy_a_delta(pcm.data(), dst.data(), (int64_t)C * S);
        rep->encode_seconds = secs; rep->overfull = overfull;
    }
    return 0;
}

extern "C" int gsch_encode_file(const char *wav, const char *gscp, const gsch_options *o, gsch_report *rep) {
    if (!wav || !gscp || !o) return fail("gsch_encode_file: bad arguments");
    if (o->precision <= 0) return fail("-pr0 (\"lossless\" mode) writes no .gsc in the reference (enc:2021-2023)");
    int16_t *pcm = nullptr; int C = 0, sr = 0; int64_t S = 0;
    if (gsch_load_wav(wav, &pcm, &C, &S, &sr)) return 1;
    uint8_t *blob = nullptr; int64_t n = 0;
    int rc = gsch_encode_pcm(pcm, S, C, S, sr, o, &blob, &n, rep);
    free(pcm);
    if (rc) return rc;
    FILE *f = fopen(gscp, "wb");
    if (!f) { free(blob); return fail("cannot create %s", gscp); }
    fwrite(blob, 1, (size_t)n, f);
    fclose(f);
    free(blob);
    return 0;
}

extern "C" int gsch_decode_file(const char *gscp, const char *wav) {
    FILE *f = fopen(gscp, "rb");
    if (!f) return fail("cannot open %s", gscp);
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    std::vector<uint8_t> g((size_t)std::max(n, 1L));
    if (n > 0 && fread(g.data(), 1, (size_t)n, f) != (size_t)n) { fclose(f); return fail("%s: short read", gscp); }
    fclose(f);
    int C = 0, sr = 0;
    const int64_t S = gsch_decode(g.data(), n, nullptr, 0, &C, &sr);
    if (S < 0) return fail("%s: malformed .gsc stream", gscp);
    std::vector<int16_t> out((size_t)std::max<int64_t>(S, 1) * std::max(C, 1));
    gsch_decode(g.data(), n, out.data(), S, &C, &sr);
    return gsch_save_wav(wav, out.data(), C, S, sr);
}
