// gsc_encode -- command-line encoder with the reference's interface (enc:1939-2056):
//     gsc_encode <source.wav> <dest.gsc> [options]
// Host steps from libgsc_host.so, DoFrame on the GPU(s) through libgsc_cuda.so.
#include <cstdio>
#include <cstring>
#include <string>

#include "../include/gsc_host.h"

static void usage(const char *argv0) {   // enc:1957-1981
    printf("Usage: %s <source file> <dest file> [options]\n", argv0);
    printf("Main options:\n");
    printf("\t-br\tencoder bit rate in kilobits/second; example: \"-br250\"\n");
    printf("\t-vfr\tRMS power based variable frame size ratio (0.0-1.0); default: \"-vfr1.0\"\n");
    printf("\t-fl\t(Average) frame length in milliseconds; default: \"-fl4000\"\n");
    printf("\t-v\tverbose mode\n");
    printf("Development options:\n");
    printf("\t-cs\tchunk size\n");
    printf("\t-cpf\tmax. chunks per frame (256-4096)\n");
    printf("\t-cbd\tchunk bit depth (8,12)\n");
    printf("\t-pr\tK-means precision\n");
    printf("GPU options (not in the reference):\n");
    printf("\t-gpus\tnumber of GPUs to shard frames over (default: all)\n");
    printf("\t-lloyd\tbatch Lloyd with the given iteration count instead of the reference's online rule\n");
    printf("\t-kdtree\tsearch through the reference's ANN kd-tree (its encoder's output; -cs2 and -cs4)\n");
    printf("\n(source file must be 16bit WAV)\n\n");
}

int main(int argc, char **argv) {
    if (argc < 3) { usage(argv[0]); return 0; }
    gsch_options o;
    gsch_default_options(&o);
    for (int i = 3; i < argc; ++i)
        if (gsch_parse_option(&o, argv[i])) { fprintf(stderr, "unknown or unsupported option %s\n", argv[i]); return 2; }
    printf("BitRate = %d\nVariableFrameSizeRatio = %g\nFrameLength = %.0f\n", o.bitrate, o.vfr, o.frame_length_ms);
    if (o.verbose)
        printf("ChunkSize = %d\nMaxChunksPerFrame = %d\nChunkBitDepth = %d\nPrecision = %d\n", o.chunk_size, o.chunks_per_frame,
               o.chunk_bit_depth, o.precision);
    std::string dst = argv[2];   // enc:1188 ChangeFileExt(outputFN, '.gsc')
    size_t dot = dst.find_last_of('.'), slash = dst.find_last_of('/');
    if (dot != std::string::npos && (slash == std::string::npos || dot > slash)) dst.erase(dot);
    dst += ".gsc";
    printf("Load %s\n", argv[1]);
    gsch_report r;
    memset(&r, 0, sizeof(r));
    if (gsch_encode_file(argv[1], dst.c_str(), &o, &r)) { fprintf(stderr, "error: %s\n", gsch_last_error()); return 1; }
    printf("ChannelCount = %d\nSampleRate = %d\nFrameCount = %d\nChunksPerFrame = %d\n", r.channels, r.sample_rate, r.frames,
           r.chunks_per_frame);
    printf("Save %s\nFinalByteSize = %lld\nFinalBitRate = %.0f\n", dst.c_str(), (long long)r.gsc_bytes, r.bitrate_kbps);
    printf("PsyADelta = %.10f\n", r.psy_a_delta);
    printf("GPUs = %d\nMakeFrames seconds = %.3f (%.1fx real time)\n", r.devices, r.encode_seconds,
           ((double)r.samples / r.sample_rate) / (r.encode_seconds > 0 ? r.encode_seconds : 1e-9));
    if (r.overfull) printf("note: %lld queries had more than 64 rows inside the epsilon band (ANN truncation not reproduced)\n", (long long)r.overfull);
    return 0;
}
