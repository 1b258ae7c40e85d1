/*
 * jpgenc_b200.h — C-ABI of the B200-native JPEG encode path that drops in behind Nuos/jpgEnc's C++ surface.
 *
 * The reference has no FFI: its "interface" for this path is the stage methods of `class Image`
 * (reference include/Image.hpp:76-92) driven by Image::writeJPEG (reference src/Image.cpp:831-976).
 * Each entry point below names the reference code it replaces.  Plain pointers and sizes only; no
 * exceptions cross this boundary: every call returns JPGENC_OK (0) or a negative code and
 * jpgenc_last_error() gives the text.  The C++ host mirror (jpgenc_b200/host/) rethrows failures as
 * std::runtime_error, which is what the reference throws (src/Image.cpp:428,450).
 *
 * Ownership: the caller owns every host pointer; the context owns all device memory and one CUDA
 * stream.  Threading: one context per host thread / GPU; independent contexts may run concurrently
 * (this is how a batch of images is sharded over GPUs).  There is no CPU fallback: without a CUDA
 * device jpgenc_create fails.
 *
 * Device layouts (DESIGN.md "Data layout in HBM"):
 *   rgb     u8  interleaved R,G,B, real_w*real_h*3, exactly the P6 payload (src/Image.cpp:411-418)
 *   coef    i16 MCU-ordered: per 16x16 MCU the blocks Y00,Y01,Y10,Y11,Cb,Cr (the order of
 *           src/Image.cpp:959-967), 64 coefficients each in ZIGZAG order, DC not differenced
 *   scan    u8  entropy-coded segment: MCU-interleaved, 1-padded, FF->FF00 stuffed
 */
#ifndef JPGENC_B200_H
#define JPGENC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JPGENC_OK             0
#define JPGENC_ERR_CUDA      -1   /* a CUDA runtime call failed (text in jpgenc_last_error) */
#define JPGENC_ERR_ARG       -2   /* bad argument / call out of pipeline order */
#define JPGENC_ERR_NO_DEVICE -3   /* no usable CUDA device: there is no CPU fallback */
#define JPGENC_ERR_FORMAT    -4   /* not a P3/P6 PPM (reference: std::runtime_error, src/Image.cpp:449-450) */
#define JPGENC_ERR_IO        -5   /* file could not be opened (reference: src/Image.cpp:427-428) */
#define JPGENC_ERR_CAPACITY  -6   /* caller's output buffer too small */
#define JPGENC_ERR_NOMEM     -7   /* host memory exhausted (a C++ exception was caught at the boundary; text in jpgenc_last_error) */

/* Pixel formats of the *_image calls.  A 4th byte is never read into the image and takes no part in the maxval check.
 * Together with a row pitch (bytes from one row to the next; 0 = width * bytes per pixel, never less than that) they describe
 * the pixels only: the file is the one the reference writes for the same R,G,B samples. */
#define JPGENC_PIXEL_RGB      0   /* 3 bytes per pixel: R,G,B */
#define JPGENC_PIXEL_BGR      1   /* 3 bytes per pixel: B,G,R */
#define JPGENC_PIXEL_RGBA     2   /* 4 bytes per pixel: R,G,B, then a byte that is ignored */
#define JPGENC_PIXEL_BGRA     3   /* 4 bytes per pixel: B,G,R, then a byte that is ignored */
#define JPGENC_PIXEL_GRAY    16   /* 1 byte per pixel v, encoded as the pixel (v, v, v): the reference's file for that RGB image */

typedef struct jpgenc_ctx jpgenc_ctx;

/* Table ids everywhere: 0 = Y_DC, 1 = Y_AC, 2 = C_DC, 3 = C_AC (src/Image.cpp:908-912, 946-949). */
typedef struct {
    uint32_t code_msb[256];   /* Code::code, MSB-aligned (include/Huffman.hpp:21-46) */
    uint8_t  length[256];     /* 0 = symbol absent */
    uint8_t  counts[16];      /* DHT: codes per length 1..16 (JpegSegments.hpp:188-218) */
    uint8_t  symbols[256];    /* DHT: symbols in the reference's SymbolsPerLength order */
    int32_t  nsymbols;
} jpgenc_huff_table;

typedef struct {
    uint32_t real_w, real_h;      /* as in the PPM header */
    uint32_t mcu_w, mcu_h;        /* padded to x16 (src/Image.cpp:479-489) */
    uint64_t n_blocks;            /* mcu_w*mcu_h*6 */
    uint64_t refined_blocks;      /* blocks re-done in exact FP64 because an FP32 quotient sat on a rounding boundary */
    uint64_t scan_bits;           /* entropy-coded bits before padding */
    uint64_t scan_bytes;          /* after 1-padding and FF00 stuffing */
    uint64_t stuffed_ff;          /* number of 0xFF bytes that received a 0x00 */
    /* stage times: 0 unless jpgenc_set_stage_timing has switched the event records on (level 1: ms_k1; level 2: all four) */
    float    ms_k1;               /* CUDA-event time of the last K1 fast kernel alone (the roofline kernel) */
    float    ms_forward;          /* CUDA-event time of the last K1 + exact refinement */
    float    ms_stats;            /* last K2 */
    float    ms_entropy;          /* last K3 + K4 */
    float    ms_h2d, ms_d2h;      /* the copies of the calls that take or return host memory (always measured) */
    /* running sums of the four stage times over every whole-image encode on this context since it was created, and their
     * number: a caller that times many encodes reads them once before and once after instead of polling every encode */
    double   sum_ms_k1, sum_ms_forward, sum_ms_stats, sum_ms_entropy;
    uint64_t timed_encodes;
} jpgenc_stats;

/* ---- lifecycle ------------------------------------------------------------------------------------ */
int  jpgenc_create(int device, jpgenc_ctx** out);
/* CUDA-event records between the kernels of a single image, for jpgenc_stats' stage times: level 0 (the default) none,
 * 1 around the K1 fast kernel alone, 2 around every stage.  They are not free: inside the replayed graphs of a single
 * image every record is a node of its own, about 3 us each (3840x2160 frame: 0.092 ms without, 0.115 ms with all eight). */
int  jpgenc_set_stage_timing(jpgenc_ctx* ctx, int level);
void jpgenc_destroy(jpgenc_ctx* ctx);
/* ctx may be NULL: text of the last failure of jpgenc_create on this thread */
const char* jpgenc_last_error(const jpgenc_ctx* ctx);
/* the context's cudaStream_t, so a caller can record its own CUDA events around the stage calls */
void* jpgenc_stream(jpgenc_ctx* ctx);
int  jpgenc_synchronize(jpgenc_ctx* ctx);
int  jpgenc_get_stats(jpgenc_ctx* ctx, jpgenc_stats* out);

/* ---- parameters the reference hard-codes in writeJPEG --------------------------------------------- */
/* natural (row-major) order, as in src/Image.cpp:850-869; defaults are those Annex-K tables */
int jpgenc_set_qtables(jpgenc_ctx* ctx, const uint8_t qy[64], const uint8_t qc[64]);
/* AAN constants a1..a5, s0..s7 evaluated by the HOST with the reference's expressions
 * (include/Dct.hpp:21-43) so the exact path uses bit-identical doubles; optional (the library computes
 * the same expressions itself when this is never called) */
int jpgenc_set_dct_constants(jpgenc_ctx* ctx, const double a[5], const double s[8]);

/* ---- input: replaces loadPPM's pixel path (src/Image.cpp:411-418, 465, 479-532) -------------------- */
/* H2D of raw samples (P6 payload or parsed P3), maxval < 256.  Scaling by 255/maxval and the x16
 * edge-replication padding happen on the device.  host_rgb should be pinned for full PCIe speed.
 * Contract: every sample <= maxval.  Host pixels are checked when maxval < 255 (JPGENC_ERR_FORMAT; the PPM readers refuse such
 * files the same way): the reference would scale such a sample past 255, which the 8-bit path's exactness thresholds do not
 * cover -- jpgenc_encode_planes takes that kind of data.  Device-resident pixels (bind, frames) are the caller's promise. */
int jpgenc_upload_rgb(jpgenc_ctx* ctx, const uint8_t* host_rgb, uint32_t real_w, uint32_t real_h, uint32_t maxval);
/* same, for pixels that already live in device memory (no copy is made; the pointer must stay valid) */
int jpgenc_bind_device_rgb(jpgenc_ctx* ctx, const void* dev_rgb, uint32_t real_w, uint32_t real_h, uint32_t maxval);
/* same, for device pixels in any JPGENC_PIXEL_* format with a row pitch (0 = tight); crops of a larger image and pitched
 * allocations are read where they are.  Then jpgenc_color_dct_quant / jpgenc_encode_bound as after jpgenc_bind_device_rgb.
 * Unknown format, pitch below the row size, sides outside 1..65535: JPGENC_ERR_ARG. */
int jpgenc_bind_device_image(jpgenc_ctx* ctx, const void* dev, uint32_t real_w, uint32_t real_h, uint32_t row_pitch, int format,
                             uint32_t maxval);
/* same, for planar RGB: one plane of 1 byte per pixel per channel, the three with one row pitch (0 = real_w).  BGR or GBR plane
 * order is a different assignment of the pointers; planes may alias (r == g == b gives the JPGENC_PIXEL_GRAY file).
 * A null plane, pitch below real_w, sides outside 1..65535: JPGENC_ERR_ARG. */
int jpgenc_bind_device_planar(jpgenc_ctx* ctx, const void* r, const void* g, const void* b, uint32_t real_w, uint32_t real_h,
                              uint32_t row_pitch, uint32_t maxval);
/* YUV 4:2:0 frames with 8-bit samples, as video decoders leave them.  A w x h frame has a Y plane of h rows of w bytes, y_pitch
 * apart (0 = w), and chroma planes of ch = ceil(h/2) rows of cw = ceil(w/2) samples, c_pitch apart:
 *   JPGENC_YUV_I420: U and V planes of cw bytes per row (0 = cw); YV12 is I420 with the u and v pointers swapped;
 *   JPGENC_YUV_NV12: one plane of cw (U, V) byte pairs per row (0 = 2 cw), passed as u; v must be NULL.
 * The samples are the file's Y, Cb and Cr as they are (JFIF reads them as full-range BT.601; no range or matrix conversion is
 * done, and there is no maxval): the file is jpgenc_encode_planes(..., ycbcr = 1) of the planes Y - 128, Cb - 128, Cr - 128
 * with every chroma sample repeated over its 2x2 pixels and the frame padded to whole MCUs by edge replication -- the
 * reference's own 4:2:0 file of that YCbCr image, byte for byte.  Then jpgenc_color_dct_quant / jpgenc_encode_bound as after
 * any other bind.  Unknown layout, a null Y or U plane, a null V plane for I420 or a non-null one for NV12, a pitch below its
 * row size, sides outside 1..65535: JPGENC_ERR_ARG. */
#define JPGENC_YUV_I420 0   /* Y, U, V planes */
#define JPGENC_YUV_NV12 1   /* Y plane, interleaved UV plane (passed as u; v must be NULL) */
int jpgenc_bind_device_yuv420(jpgenc_ctx* ctx, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                              uint32_t c_pitch, int layout);
/* YUV frames with 8-bit samples in any of these layouts (and the two above), as cameras, capture cards and decoders leave them.
 * With cw = ceil(w/2), a frame has:
 *   JPGENC_YUV_I422: a Y plane of h rows of w bytes, U and V planes of h rows of cw bytes, c_pitch apart (0 = cw); YV16 is I422
 *                    with the u and v pointers swapped (ffmpeg yuv422p / yuvj422p);
 *   JPGENC_YUV_NV16: a Y plane and one plane of h rows of cw (U, V) byte pairs (0 = 2 cw), passed as u; v must be NULL;
 *   JPGENC_YUV_I444: Y, U and V planes of h rows of w bytes; U and V share c_pitch (0 = w) (ffmpeg yuv444p);
 *   JPGENC_YUV_YUYV: one packed plane of h rows of cw groups Y0 U Y1 V (4 cw bytes, y_pitch apart; V4L2_PIX_FMT_YUYV), passed as
 *                    y; u and v must be NULL and c_pitch 0.  For an odd w the second Y of the last group is never read;
 *   JPGENC_YUV_UYVY: the same with groups U Y0 V Y1 (8-bit YUV of SDI capture cards).
 * The colour contract is that of the 4:2:0 layouts: the samples are the file's Y, Cb and Cr as they are.  The file is always the
 * reference's 4:2:0 file: jpgenc_encode_planes(..., ycbcr = 1) of the planes Y - 128, U - 128, V - 128 at full resolution
 * (every 4:2:2 chroma sample repeated over its two pixels), padded to whole MCUs by edge replication -- so the chroma of a 2x2
 * cell is the mean of its four (clamped) samples, as S420_m takes it.  These three calls take all seven JPGENC_YUV_* codes;
 * jpgenc_bind_device_yuv420 / jpgenc_encode_yuv420 / jpgenc_encode_images_packed_yuv420 only the two 4:2:0 ones.  Unknown
 * layout, a null Y plane, a null chroma plane where one is needed or a non-null one where it must be NULL, c_pitch != 0 for the
 * packed layouts, a pitch below its row size, sides outside 1..65535: JPGENC_ERR_ARG. */
#define JPGENC_YUV_I422 2   /* Y, U, V planes, chroma of cw x h */
#define JPGENC_YUV_NV16 3   /* Y plane, interleaved UV plane of cw pairs x h (passed as u; v must be NULL) */
#define JPGENC_YUV_I444 4   /* Y, U, V planes, all w x h */
#define JPGENC_YUV_YUYV 5   /* one packed plane of Y0 U Y1 V groups (passed as y) */
#define JPGENC_YUV_UYVY 6   /* one packed plane of U Y0 V Y1 groups (passed as y) */
int jpgenc_bind_device_yuv(jpgenc_ctx* ctx, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                           uint32_t c_pitch, int layout);

/* ---- K1: convertToColorSpace(YCbCr) + applySubsampling(S420_m) + applyDCT(Arai) + applyQuantization
 *      + zigzag (src/Image.cpp:112-148, 198-235, 540-595, 597-636; Dct.hpp:47-215; Coding.hpp:57-97) -- */
int jpgenc_color_dct_quant(jpgenc_ctx* ctx);
/* test hooks: read the coefficients back (n_blocks*64 int16, MCU order) / feed the REFERENCE's planar
 * natural-order int32 arrays QY,QCb,QCr (Image.hpp:112) so K2-K4 can be checked independently of K1 */
int jpgenc_get_coefficients(jpgenc_ctx* ctx, int16_t* dst);
int jpgenc_set_coefficients(jpgenc_ctx* ctx, const int32_t* q_y, const int32_t* q_cb, const int32_t* q_cr,
                            uint32_t mcu_w, uint32_t mcu_h);
/* feed MCU-ordered zigzag int16 coefficients directly */
int jpgenc_set_coefficients_mcu(jpgenc_ctx* ctx, const int16_t* coef, uint32_t mcu_w, uint32_t mcu_h);

/* ---- K2: applyDCdifferenceCoding + doRLEandCategoryCoding + the symbol texts
 *      (src/Image.cpp:638-735, 888-906; Coding.hpp:148-283) reduced to what the table build needs ----- */
/* count[t][s] = occurrences of symbol s in table t's text; first_pos[t][s] = an order-preserving key of
 * its first occurrence in that text (UINT64_MAX if absent): (block index in text order)*256 + k with k = 0 for a DC
 * symbol, 2p for a ZRL emitted before zigzag position p, 2p+1 for the symbol of position p, 129 for EOB */
int jpgenc_symbol_stats(jpgenc_ctx* ctx, uint32_t count[4][256], uint64_t first_pos[4][256]);

/* ---- host: generateHuffmanCode from the statistics (src/Huffman.cpp:3-66, Huffman.hpp:114-174) ----- */
int jpgenc_build_huffman(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out);
/* the same tables from the plain statement of the algorithm (one std container per container of the reference, one vector
 * per package-merge level): the anchor jpgenc_build_huffman (allocation-free queues) and the device build are tested against */
int jpgenc_build_huffman_containers(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out);

/* the same on the device, n tables at once (one warp per table; libstdc++'s container orders restated on arrays).  The
 * batched-frame calls use it when the process has few host cores for its GPU (8-GPU boxes); identical results. */
/* the device build's code run on the HOST (no GPU): the array restatement against the container-driven build, for the
 * CPU test suite */
int jpgenc_build_huffman_arrays(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out);
int jpgenc_build_huffman_device(jpgenc_ctx* ctx, uint32_t n, const uint32_t (*count)[256], const uint64_t (*first_pos)[256],
                                jpgenc_huff_table* out);

/* ---- K3 + K4: doHuffmanEncoding, MCU interleave, fill(), FF00 stuffing
 *      (src/Image.cpp:737-829, 957-971; BitstreamGeneric.hpp:182-195, 213-224, 242-248) ------------- */
int jpgenc_entropy_encode(jpgenc_ctx* ctx, const jpgenc_huff_table tables[4], uint64_t* scan_bytes);
int jpgenc_download_scan(jpgenc_ctx* ctx, uint8_t* dst, uint64_t cap);

/* ---- host: PPM front end with the reference's parsing rules (src/Image.cpp:334-473); no GPU involved ---- */
/* header of a P3/P6 file held in memory; returns JPGENC_ERR_FORMAT for anything else */
int jpgenc_ppm_info(const uint8_t* file, size_t n, uint32_t* width, uint32_t* height, uint32_t* maxval, int* magic,
                    size_t* payload_offset);
/* raw samples (NOT scaled by 255/maxval) as interleaved u8 RGB; dst holds width*height*3 bytes */
int jpgenc_ppm_samples(const uint8_t* file, size_t n, uint8_t* dst);

/* ---- whole image: what Image::writeJPEG does after loadPPM ----------------------------------------- */
/* headers SOI..SOS (src/Image.cpp:933-954, JpegSegments.hpp); returns the length, dst may be NULL */
size_t jpgenc_write_headers(uint32_t real_w, uint32_t real_h, const uint8_t qy[64], const uint8_t qc[64],
                            const jpgenc_huff_table tables[4], uint8_t* dst);
/* runs K1..K4 on the pixels bound/uploaded and assembles headers + scan + EOI into dst */
int jpgenc_encode_bound(jpgenc_ctx* ctx, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* headers + scan of the LAST jpgenc_encode_bound on this context + EOI into dst, without re-running the pipeline */
int jpgenc_assemble_last(jpgenc_ctx* ctx, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* upload + encode (host pixels in, JPEG bytes out).  Sides outside 1..65535: JPGENC_ERR_ARG. */
int jpgenc_encode_rgb(jpgenc_ctx* ctx, const uint8_t* host_rgb, uint32_t real_w, uint32_t real_h, uint32_t maxval,
                      uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* the same for host pixels in any JPGENC_PIXEL_* format with a row pitch (0 = tight).  The rows travel as they are, in their
 * own format, the pitch gap dropped by the copy engine, and the device reads that format: no host core repacks them, and
 * 4-byte pixels cost 4/3 of the PCIe bytes of RGB.  Checked against maxval when it is below 255 (colour bytes only). */
int jpgenc_encode_image(jpgenc_ctx* ctx, const void* host, uint32_t real_w, uint32_t real_h, uint32_t row_pitch, int format,
                        uint32_t maxval, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* the same for planar RGB in host memory (see jpgenc_bind_device_planar): every plane travels as it is, one copy per plane and
 * band (one for all three when they lie back to back, as in a tight (3, H, W) buffer).  Checked against maxval when it is below
 * 255, in all three planes. */
int jpgenc_encode_planar(jpgenc_ctx* ctx, const void* r, const void* g, const void* b, uint32_t real_w, uint32_t real_h,
                         uint32_t row_pitch, uint32_t maxval, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* the same for a YUV 4:2:0 frame in host memory (see jpgenc_bind_device_yuv420): every plane travels as it is, 1.5 bytes per
 * pixel in all, the pitch gaps dropped by the copy engine; the upload of each band of MCU rows overlaps the kernels of the
 * bands before it. */
int jpgenc_encode_yuv420(jpgenc_ctx* ctx, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                         uint32_t c_pitch, int layout, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* the same for a frame in any JPGENC_YUV_* layout (see jpgenc_bind_device_yuv): 4:2:2 travels at 2 bytes per pixel, 4:4:4 at 3 */
int jpgenc_encode_yuv(jpgenc_ctx* ctx, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                      uint32_t c_pitch, int layout, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* Image::writeJPEG (src/Image.cpp:831-976) for an image given as the reference holds it: three row-major planes of doubles
 * (Image::R/G/B, include/Image.hpp:104-114), `width` x `height` = the image padded to whole 16x16 MCUs (src/Image.cpp:479-530),
 * real_w x real_h = what SOF0 reports.  ycbcr != 0: the planes already are level-shifted Y, Cb, Cr and are not converted
 * (convertToColorSpace returns at once for them, src/Image.cpp:112-115).  Any double is accepted (edited planes, non-integral
 * samples): every block is computed in FP64 in the reference's operation order.  Slower than the 8-bit path (~6 ms for 268 Mpx). */
int jpgenc_encode_planes(jpgenc_ctx* ctx, const double* p0, const double* p1, const double* p2, uint32_t width, uint32_t height,
                         uint32_t real_w, uint32_t real_h, int ycbcr, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes);
/* main.cpp:8-32 — PPM file in, JPEG file out */
int jpgenc_encode_ppm_file(jpgenc_ctx* ctx, const char* ppm_path, const char* jpg_path);

/* ---- batches: independent images on one GPU (what a caller looping over Image::writeJPEG gets, SURVEY.md 8e) ------ */
/* `workers` contexts on `device`, driven by as many host threads; frames are handed out dynamically.  Outputs are
 * byte-identical to encoding the frames one by one. */
typedef struct jpgenc_batch jpgenc_batch;
int  jpgenc_batch_create(int device, int workers, jpgenc_batch** out);
void jpgenc_batch_destroy(jpgenc_batch* batch);
const char* jpgenc_batch_last_error(const jpgenc_batch* batch);
int  jpgenc_batch_set_qtables(jpgenc_batch* batch, const uint8_t qy[64], const uint8_t qc[64]);
/* n frames of w x h interleaved RGB in host memory (pinned for full PCIe speed); out[i] (capacity caps[i]) receives
 * the complete JFIF file of frame i, sizes[i] its length.  Returns the first error (text in jpgenc_batch_last_error). */
int jpgenc_batch_encode(jpgenc_batch* batch, uint32_t n, const uint8_t* const* frames, uint32_t w, uint32_t h,
                        uint32_t maxval, uint8_t* const* out, const uint64_t* caps, uint64_t* sizes);
/* same for frames that already live in device memory; out may be NULL (scans stay on the device, sizes are reported) */
int jpgenc_batch_encode_device(jpgenc_batch* batch, uint32_t n, const void* const* dev_frames, uint32_t w, uint32_t h,
                               uint32_t maxval, uint8_t* const* out, const uint64_t* caps, uint64_t* sizes);

/* all frames TOGETHER through every kernel on one context: the batch is cut into passes of 64-128 Mpx-sized groups of frames,
 * each pass one asynchronous chain K1 > K2 > device table build > device sizes/offsets > K3 > K4 with ONE host wait (the 4*n
 * Huffman tables are built on the device, same tables as jpgenc_build_huffman), the passes rotating over four streams driven
 * by the calling thread alone.  Frames must have one size and live in device memory; out may be NULL (sizes only).  Results
 * are byte-identical to encoding the frames one by one. */
int jpgenc_encode_frames_device(jpgenc_ctx* ctx, uint32_t n, const void* const* dev_frames, uint32_t w, uint32_t h,
                                uint32_t maxval, uint8_t* const* out, const uint64_t* caps, uint64_t* sizes);
/* the same for frames in host memory (pinned for full PCIe speed): uploads of the next slice of the batch overlap the
 * kernels of the current one */
int jpgenc_encode_frames(jpgenc_ctx* ctx, uint32_t n, const uint8_t* const* frames, uint32_t w, uint32_t h,
                         uint32_t maxval, uint8_t* const* out, const uint64_t* caps, uint64_t* sizes);

/* The same batch with the output as the reference's file writer would leave it on disk, one file after the other
 * (src/Image.cpp:933-972 per frame): the complete JFIF files -- SOI..SOS headers, stuffed scan, EOI -- are assembled ON THE
 * DEVICE back to back and every pass of the batch comes home with ONE device-to-host copy into `out` (pinned for full PCIe
 * speed; `cap` bytes).  File i occupies out[offsets[i] .. offsets[i] + sizes[i]); files are in frame order without gaps,
 * *total_bytes (optional) is the end of the last one.  frames_on_device: 0 = host pointers (uploads overlap the kernels),
 * 1 = device pointers.  out may be NULL: nothing is copied, offsets/sizes are still reported. */
int jpgenc_encode_frames_packed(jpgenc_ctx* ctx, uint32_t n, const void* const* frames, int frames_on_device, uint32_t w,
                                uint32_t h, uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes,
                                uint64_t* total_bytes);

/* n images of individual sizes widths[i] x heights[i] (interleaved RGB, tightly packed rows), in host memory
 * (images_on_device = 0; pinned for full PCIe speed) or device memory (1), through the same pass pipeline: output as
 * jpgenc_encode_frames_packed -- the complete JFIF files back to back in input order in `out` (cap bytes; NULL = sizes and
 * offsets only), file i at out[offsets[i] .. offsets[i] + sizes[i]), *total_bytes (optional) the end of the last one.  Every
 * file is byte-identical to encoding that image alone.  One maxval and the context's quantisation tables apply to all images.
 * Sides are 1..65535 (JPGENC_ERR_ARG otherwise).  Host images are checked against maxval when it is below 255
 * (JPGENC_ERR_FORMAT); device images are the caller's promise.  n = 0 is legal and touches nothing.  When every image has the
 * same size this is jpgenc_encode_frames_packed. */
int jpgenc_encode_images_packed(jpgenc_ctx* ctx, uint32_t n, const void* const* images, int images_on_device, const uint32_t* widths,
                                const uint32_t* heights, uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets,
                                uint64_t* sizes, uint64_t* total_bytes);
/* jpgenc_encode_images_packed for pixels in one JPGENC_PIXEL_* format per call and a row pitch per image (row_pitches may be
 * NULL: all tight; an entry of 0 is tight too).  Tiles of one large image are pointers into it with its pitch.  Host images
 * are uploaded in their own format as in jpgenc_encode_image.  Tight RGB is jpgenc_encode_images_packed itself; every other
 * call runs the pass pipeline of images of individual sizes, equal sizes included. */
int jpgenc_encode_images_packed_layout(jpgenc_ctx* ctx, uint32_t n, const void* const* images, int images_on_device,
                                       const uint32_t* widths, const uint32_t* heights, const uint32_t* row_pitches, int format,
                                       uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes,
                                       uint64_t* total_bytes);
/* jpgenc_encode_images_packed_layout for planar RGB: planes[3i], planes[3i + 1], planes[3i + 2] are the R, G and B planes of
 * image i, row_pitches[i] their common row pitch (row_pitches may be NULL: all tight; an entry of 0 is tight too). */
int jpgenc_encode_images_packed_planar(jpgenc_ctx* ctx, uint32_t n, const void* const* planes, int images_on_device,
                                       const uint32_t* widths, const uint32_t* heights, const uint32_t* row_pitches, uint32_t maxval,
                                       uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes);
/* jpgenc_encode_images_packed_layout for YUV 4:2:0 frames of one layout (see jpgenc_bind_device_yuv420): planes[3i],
 * planes[3i + 1], planes[3i + 2] are Y, U and V of image i (NV12: Y, UV, NULL), y_pitches[i] / c_pitches[i] its pitches (either
 * array may be NULL: all tight; an entry of 0 is tight too).  Host frames are uploaded plane by plane in tight rows. */
int jpgenc_encode_images_packed_yuv420(jpgenc_ctx* ctx, uint32_t n, const void* const* planes, int images_on_device,
                                       const uint32_t* widths, const uint32_t* heights, const uint32_t* y_pitches,
                                       const uint32_t* c_pitches, int layout, uint8_t* out, uint64_t cap, uint64_t* offsets,
                                       uint64_t* sizes, uint64_t* total_bytes);
/* the same for frames in any JPGENC_YUV_* layout (see jpgenc_bind_device_yuv), one layout per call: planes[3i .. 3i + 2] are
 * Y, U, V of frame i (NV12 / NV16: Y, UV, NULL; YUYV / UYVY: the packed plane, NULL, NULL) */
int jpgenc_encode_images_packed_yuv(jpgenc_ctx* ctx, uint32_t n, const void* const* planes, int images_on_device,
                                    const uint32_t* widths, const uint32_t* heights, const uint32_t* y_pitches,
                                    const uint32_t* c_pitches, int layout, uint8_t* out, uint64_t cap, uint64_t* offsets,
                                    uint64_t* sizes, uint64_t* total_bytes);

/* ---- stage methods for the modes writeJPEG does not use (SURVEY.md 8(f)4) ------------------------------------------ */
/* Image::applySubsampling(mode) on one chroma plane (src/Image.cpp:198-319): `plane` = height x width doubles (host), mode =
 * the order of Image::SubsamplingMode (0 S444, 1 S422, 2 S411, 3 S420, 4 S420_m, 5 S420_lm); `out` receives the
 * (height / vdiv) x (width / hdiv) plane (jpgenc_stage_subsample_dims).  Same doubles as the reference, bit for bit. */
int jpgenc_stage_subsample_dims(int mode, uint32_t width, uint32_t height, uint32_t* out_width, uint32_t* out_height);
int jpgenc_stage_subsample(jpgenc_ctx* ctx, const double* plane, uint32_t width, uint32_t height, int mode, double* out);
/* Image::applyDCT(mode) on one plane (src/Image.cpp:540-595): every 8x8 block through dctDirect / dctMat / dctArai
 * (include/Dct.hpp:238-262, 264-276, 47-215; mode 0 Simple, 1 Matrix, 2 Arai = the order of Image::DCTMode).  `plane` and `out`:
 * height x width doubles (host), sides multiples of 8.  Same doubles as the reference, bit for bit. */
int jpgenc_stage_dct(jpgenc_ctx* ctx, const double* plane, uint32_t width, uint32_t height, int mode, double* out);

/* ---- config-1 microbenchmark: dctArai + quantize + zigzag on stand-alone blocks -------------------- */
/* dev_in: nblocks*64 fp32 samples (row-major 8x8 per block); dev_out: nblocks*64 int16 zigzag.
 * Same exactness contract as K1 (FP32 fast path + exact FP64 refinement of boundary cases). */
int jpgenc_dct_quant_blocks(jpgenc_ctx* ctx, const float* dev_in, int16_t* dev_out, uint64_t nblocks,
                            const uint8_t q[64], uint64_t* refined_blocks);

/* ---- deployment helper: one process per GPU on a multi-socket host ------------------------------------------------- */
/* Restricts the calling thread to the CPUs of the NUMA node `device` is attached to (sysfs), so that pinned buffers it
 * allocates afterwards are node-local and its uploads do not cross the socket interconnect.  *numa_node = that node, or
 * -1 when the topology is unknown or the node's CPUs are not available to the process (then nothing is changed);
 * *cpus_bound = CPUs in the new mask.  Call before allocating pinned memory. */
int jpgenc_bind_host_to_device_numa(int device, int* numa_node, int* cpus_bound);

/* diagnostics for tests: one of the context's device-side counters (index 6: chunks the Huffman packer took the slow way) */
int jpgenc_debug_counter(jpgenc_ctx* ctx, int index, uint32_t* value);

/* ---- plain device-memory helpers so a Python/C harness needs no other CUDA binding ---------------- */
int jpgenc_dev_alloc(jpgenc_ctx* ctx, size_t bytes, void** dev_ptr);
int jpgenc_dev_free(jpgenc_ctx* ctx, void* dev_ptr);
int jpgenc_host_alloc_pinned(size_t bytes, void** host_ptr);
int jpgenc_host_free_pinned(void* host_ptr);
int jpgenc_memcpy_h2d(jpgenc_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes);
int jpgenc_memcpy_d2h(jpgenc_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);
/* device-side synthetic generators (SURVEY.md 8d) so benches need no multi-GB uploads */
int jpgenc_synth_rgb(jpgenc_ctx* ctx, void* dev_rgb, uint32_t w, uint32_t h, uint32_t seed);
int jpgenc_synth_blocks(jpgenc_ctx* ctx, float* dev_blocks, uint64_t nblocks);
/* write `bytes` of a scratch buffer (>= L2 size) to evict L2 between timed iterations */
int jpgenc_flush_l2(jpgenc_ctx* ctx);
/* CUDA-event timing on the context's stream: begin/end return elapsed ms of everything enqueued between */
int jpgenc_timer_begin(jpgenc_ctx* ctx);
int jpgenc_timer_end(jpgenc_ctx* ctx, float* ms);
/* number of kernels this library has launched on the context since creation */
uint64_t jpgenc_launch_count(const jpgenc_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
