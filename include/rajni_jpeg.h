/*
 * rajni_jpeg.h — C ABI of librajni_jpeg.so, the GPU JPEG decoder of the input pipeline.
 *
 * It decodes the baseline subset that covers almost all of ImageNet into the packed-frame layout that
 * rajni_resize_center_crop_u8 (rajni_b200.h) consumes, and every frame it produces equals
 * PIL.Image.open(f).convert("RGB") byte for byte (libjpeg's ISLOW IDCT, fancy upsampling and YCbCr tables;
 * oracle/jpeg_oracle.py restates the arithmetic).  What it takes:
 *   - SOF0 / SOF1 frames with 8-bit samples and Huffman coding, one scan holding every component;
 *   - 1 component (grayscale, decoded as R = G = B = Y), or 3 components libjpeg treats as YCbCr (a JFIF marker, else
 *     the Adobe transform flag, else component ids other than 'R','G','B');
 *   - luma sampling 1x1, 2x1 or 2x2 with 1x1 chroma (4:4:4, 4:2:2, 4:2:0);
 *   - up to 4 DC and 4 AC tables, 8- and 16-bit quantisation tables, restart intervals, sides up to 16384.
 * Everything else (progressive, arithmetic, 12-bit, lossless, CMYK/YCCK, RGB, other sampling, multi-scan, not a JPEG)
 * and files that do not end in an EOI marker (most truncated files) are refused by rajni_jpeg_parse and are the
 * caller's to decode on the CPU.  A stream the GPU finds malformed is reported
 * per image by rajni_jpeg_status; the caller decodes those on the CPU too, so its errors are the CPU decoder's own.
 *
 * Conventions are rajni_b200.h's: pointers are DEVICE pointers unless the name ends in _host, `stream` is a cudaStream_t
 * passed as void*, calls return RAJNI_OK or a negative RAJNI_E* code with the message in rajni_jpeg_last_error()
 * (thread-local).  The library is separate from librajni_b200.so, whose surface is the model boundary.
 */
#ifndef RAJNI_JPEG_H
#define RAJNI_JPEG_H

#include "rajni_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RAJNI_JPEG_VERSION 1

/* per-image outcome of a decode, read with rajni_jpeg_status */
enum {
    RAJNI_JPEG_OK = 0,
    RAJNI_JPEG_SKIPPED = 1,       /* info.gpu == 0: not decoded, the frame slot is the caller's to fill        */
    RAJNI_JPEG_TRUNCATED = 2,     /* the entropy-coded data ended (a marker or the end of the bytes) too early */
    RAJNI_JPEG_BAD_CODE = 3,      /* a bit pattern that no Huffman code of the table matches                 */
    RAJNI_JPEG_BAD_RUN = 4,       /* an AC run past coefficient 63                                            */
    RAJNI_JPEG_BAD_RESTART = 5    /* data before a restart marker, or not the expected RSTn                  */
};

/* Headers of one file, as rajni_jpeg_parse reads them.  Treat as opaque except for the first fields. */
typedef struct rajni_jpeg_info {
    int gpu;                       /* 1: the GPU decodes this file; 0: it does not (`why` says why)               */
    int width, height, ncomp;      /* frame size; 1 or 3 components                                               */
    int h_samp, v_samp;            /* luma sampling factors relative to chroma: 1x1, 2x1 or 2x2 (1x1 for gray)    */
    int restart_interval;          /* MCUs per restart interval, 0 = none                                         */
    long long scan_offset;         /* first byte of the entropy-coded data, from the start of the file            */
    long long file_bytes;
    int qt[3], dc[3], ac[3];       /* table ids of each component                                                 */
    unsigned short quant[4][64];   /* quantisation tables, natural order                                          */
    unsigned char huff_bits[8][16];    /* DC tables 0..3, then AC tables 0..3: code counts per length 1..16    */
    unsigned char huff_vals[8][256];
    char why[64];
} rajni_jpeg_info;

int rajni_jpeg_version(void);
const char* rajni_jpeg_last_error(void);

/* Host only (no CUDA call; safe in data-loader worker processes).  Reads the headers of the `nbytes`-byte file at
 * data_host up to its first scan and fills *info.  Returns info->gpu: 1 if the GPU decodes it, 0 if not (including bytes
 * that are not a JPEG at all, or a header cut short); never fails otherwise. */
int rajni_jpeg_parse(const void* data_host, long long nbytes, rajni_jpeg_info* info);

/* Device workspace that rajni_jpeg_decode needs for these B files (entries with gpu == 0 cost nothing). */
size_t rajni_jpeg_workspace_bytes(const rajni_jpeg_info* infos_host, int B);

/* Decode the B files on `stream`: jpeg_huffman (one decoder per image, Huffman tables in shared memory) -> int16
 * coefficients, jpeg_idct (dequantise + ISLOW) -> sample planes, jpeg_color (upsampling + YCbCr->RGB) -> frames.
 * files: the file bytes, file b at files + file_offsets_host[b] (its length is infos_host[b].file_bytes);
 * frames: output, frame b (HWC uint8, height x width x 3) written at frames + frame_offsets_host[b] for every b with
 * gpu == 1 - the layout (offset, H, W) of rajni_resize_center_crop_u8's meta.  Tables and per-image jobs are built
 * on the host and copied with one cudaMemcpyAsync. */
int rajni_jpeg_decode(const void* files, const long long* file_offsets_host, const rajni_jpeg_info* infos_host, int B,
                      void* frames, const long long* frame_offsets_host, void* workspace, size_t workspace_bytes,
                      void* stream);

/* Per-image RAJNI_JPEG_* outcome of the last decode on this workspace into status_host[B].  Synchronises the stream.
 * Returns RAJNI_OK or a negative error code. */
int rajni_jpeg_status(const void* workspace, int B, int* status_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAJNI_JPEG_H */
