/*
 * b2j.h -- C ABI of the B200-native baseline-JPEG decode path.
 *
 * This is the drop-in boundary for the hot path of xinfushe/oclJPEGDecoder
 * (entropy decode -> dequant/IDCT -> chroma upsample + YCbCr->BGRA). Plain pointers and
 * sizes only; no C++ or torch types. Everything behind it is hand-written CUDA for sm_100a.
 * There is no CPU fallback: every entry point that needs the device fails with
 * B2J_E_NODEVICE / B2J_E_CUDA when no B200 is usable.
 *
 * Which reference interface each entry point replaces (paths relative to the reference repo):
 *
 *   b2j_parse_header        parser.cpp:272-372  load_jpg() up to and including SOS, with the
 *                                               segment readers read_soi/dqt/sof/dht/dri/sos
 *                                               (parser.cpp:7-270) and the accept gate
 *                                               is_supported_file() (decoder.h:4, decoder.cpp:18-70)
 *                                               and the geometry of decode_init() (decoder.cpp:161-199)
 *   b2j_create/destroy      idct.h:9-10,18      Initialize_OpenCL_IDCT(), clidct_create(),
 *                                               clidct_clean_up() (oclDCT8x8.cpp:25-110,306-341)
 *   b2j_batch_create        idct.h:11-12        clidct_allocate_memory() + the host->device
 *                                               transfer (oclDCT8x8.cpp:112-165); here the
 *                                               COMPRESSED scan is uploaded, not coefficients
 *   b2j_batch_decode        decoder.h:6-7       decode_huffman_data() + decode_mcu_data()
 *                                               (decoder.cpp:262-365, 397-523) and clidct_run()
 *                                               (idct.h:14, oclDCT8x8.cpp:275-299)
 *   b2j_batch_decode_timed, b2j_batch_decode_steps
 *                           parser.cpp:373-397  the clock() stage timers of load_jpg(), as CUDA events
 *   b2j_batch_sync          idct.h:17           clidct_wait_for_completion()
 *   b2j_batch_read_pixels   idct.h:16           clidct_retrieve_image_from_device() (tight pitch W*4)
 *   b2j_batch_read_coefs    idct.h:15           clidct_retrieve_data_from_device(): int32[blk][64],
 *                                               natural order, dequantised == JPG_DATA::mcu_data
 *                                               after decode_huffman_data() (jpeg.h:74)
 *   b2j_decode_host(_ex)    parser.cpp:376-397  the whole per-file sequence, batched, host buffers
 *                                               in and out; _ex: output layout, host threads for parsing/staging
 *   b2j_decode_host_multi   main.cpp:17-37      one call over several GPUs: images are sharded by compressed bytes,
 *                                               one host thread and one context per GPU, no exchange between them
 *   b2j_batch_downscale     (none)              reduced copies of the decoded pixels for consumers (SURVEY.md 8f rank 3)
 *   b2j_batch_set_scale     (none)              libjpeg's scaled decode (scale_num / scale_denom, Pillow's draft()):
 *                                               1/2, 1/4 or 1/8 size straight from the coefficients
 *   b2j_parse_orientation,  (none)              EXIF orientation as OpenCV's imdecode, torchvision's decode_jpeg(...,
 *   b2j_batch_set_orientations                  apply_exif_orientation=True) and Pillow's exif_transpose() apply it
 *   b2j_batch_set_crops,    (none)              a crop window per image (SURVEY.md 8f rank 3), decoded from the MCUs
 *   b2j_decode_host_crop                        it touches: a training loader's RandomResizedCrop / CenterCrop input
 *   b2j_idct_*              idct.h:9-18         the device backend as the reference's own decoder.cpp drives it
 *                                               (coefficients in, pixels out): see "secondary boundary" below
 *   b2j_read_files          decoder.cpp:94-101  the 2 KiB fread() loop (and main.cpp's fopen): whole files read with
 *                                               several threads into one pinned arena
 *   b2j_host_alloc/free     oclDCT8x8.cpp:112-165 the host side of clidct_allocate_memory(): pinned buffers, so that
 *                                               the device<->host copies run at PCIe speed
 *
 * The C++ shim that keeps the reference's own four decoder.h signatures on top of this ABI is
 * ocljpegdecoder_b200/csrc/refshim/; INTEGRATION.md shows the binding.
 */
#ifndef B2J_H_INCLUDED
#define B2J_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2J_ABI_VERSION 5

/* ---- return codes (0 = success, like the reference's `true`) ---- */
#define B2J_OK 0
#define B2J_E_ARG (-1)         /* bad argument                                              */
#define B2J_E_FORMAT (-2)      /* container malformed; the reference would stop parsing     */
#define B2J_E_UNSUPPORTED (-3) /* rejected by the accept gate                               */
#define B2J_E_DATA (-4)        /* entropy-coded data corrupt (see per-image status bits)    */
#define B2J_E_NOMEM (-5)
#define B2J_E_CUDA (-6)        /* a CUDA call failed; b2j_last_error() has the text         */
#define B2J_E_NODEVICE (-7)    /* no usable sm_100 device: there is no CPU fallback         */

/* ---- per-image status bits written by the kernels (0 = clean decode) ---- */
#define B2J_ST_BAD_CODE 0x01      /* bit pattern is no codeword (huffman.h:304-308)          */
#define B2J_ST_RST_MISMATCH 0x02  /* RSTn out of sequence or missing (decoder.cpp:298-302)   */
#define B2J_ST_OVERRUN 0x04       /* decode ran past its data (decoder.cpp:310-314)          */
#define B2J_ST_BLOCK_OVERFLOW 0x08 /* more than 64 coefficients in a block (decoder.cpp:259) */
#define B2J_ST_DC_RANGE 0x10      /* DC category > 16 or DC predictor outside int16          */
#define B2J_ST_SEGMENT_END 0x20   /* a restart interval did not end at its marker            */
#define B2J_ST_INTERNAL 0x4000    /* a TMA tile load did not complete (never observed; guards against a hang) */
/* A restart marker that starts no restart interval ends the image's entropy-coded data: any RSTn in a file without DRI,
 * and in a file of n intervals (n - 1 markers) the n-th marker and every later one. The reference keeps such a marker's
 * Dn byte as data and decodes on, so its coefficients differ from the file's without the marker; here a decode that needs
 * bytes behind the marker flags B2J_ST_OVERRUN instead. A stray marker behind the last block (right before EOI) changes
 * nothing, as in the reference. */

/* ---- accept gate ---- */
#define B2J_GATE_REFERENCE 0 /* exactly decoder.cpp:58-69: 4:2:0 (22,11,11) and 4:4:4        */
#define B2J_GATE_EXTENDED 1  /* + every luma sampling h x v (1..4) whose chroma factors divide it, <= 10 blocks per MCU:
                              * 4:2:2 (21,11,11; BASELINE configs[3]), 4:4:0 (12), 4:1:1 (41), 14, 31, 42, ... -- the
                              * reference's CPU loops decode these as they are (decoder.cpp:429-495), only its gate
                              * refuses them -- and, beyond the reference ("only works in ?:1:1 mode", decoder.cpp:455),
                              * chroma components with several blocks per MCU (22,21,21): the same pixel replication */
/* OR-able with either gate (SURVEY.md 8f rank 1, real-world files): tolerate what load_jpg() chokes on
 * -- COM / APPn / other length-prefixed segments anywhere before SOS are skipped (parser.cpp:410-412
 * stops at them), fill FFs before a marker are skipped, tables may be redefined, 16-bit DQT entries are
 * read big-endian as the standard says (parser.cpp:81-87 does not swap). */
#define B2J_PARSE_ROBUST 2
/* OR-able (SURVEY.md 8f rank 4): one-component (grayscale) baseline frames, which the reference refuses
 * (parser.cpp:104-106, decoder.cpp:26-31). Decoded like the luma of a colour file with U = V = 0 in YUV_to_RGB32. */
#define B2J_GATE_GRAY 4

/* ---- layout of the decoded pixels on the device (b2j_batch_set_output_format) ---- */
#define B2J_OUT_BGRA 0       /* the reference's pixels: B,G,R,0 per pixel, pitch W*4 (oclDCT8x8.cpp:196, macro.h:141-145) */
#define B2J_OUT_RGB24 1      /* R,G,B bytes interleaved, pitch W*3 (SURVEY.md 8f rank 3: what image consumers want)     */
#define B2J_OUT_RGB_PLANAR 2 /* three planes R, G, B of W*H bytes each (a CHW uint8 tensor left on the device)          */
#define B2J_OUT_GRAY8 3      /* one byte per pixel, pitch W (at the batch's scale: ceil(W/s) x ceil(H/s) bytes). Needs
                              * B2J_PIXELS_LIBJPEG. It is libjpeg's out_color_space = JCS_GRAYSCALE: the luma component's
                              * samples as they are (for a one-component file, that file's samples), with no chroma
                              * upsampling and no colour conversion; at 1/2, 1/4 and 1/8 the reduced luma IDCT's samples.
                              * The same pixels as Pillow's Image.draft("L", size), OpenCV's IMREAD_GRAYSCALE and
                              * IMREAD_REDUCED_GRAYSCALE_2/4/8, and torchvision's decode_jpeg(mode=ImageReadMode.GRAY). It is
                              * not Pillow's convert("L") of the RGB decode, which computes luminance from R, G and B. */

/* ---- which pixels a decode computes from the coefficients (b2j_batch_set_pixel_model) ---- */
#define B2J_PIXELS_REFERENCE 0 /* the reference's: Chen-Wang IDCT, chroma replication, exact integer colour (default) */
#define B2J_PIXELS_LIBJPEG 1   /* libjpeg-turbo's default decode, what Pillow, OpenCV and torchvision's CPU decoder give:
                                * ISLOW IDCT (jidctint.c), "fancy" chroma upsampling (jdsample.c: triangle filter for
                                * chroma at half the luma's width, height or both, replication for every other ratio and
                                * for chroma 1 or 2 samples wide), SCALEBITS-16 fixed-point YCbCr -> RGB (jdcolor.c).
                                * The pixels equal libjpeg-turbo's C code paths for every decodable input, and default
                                * Pillow for encoder-produced files. Caveats:
                                *  - with extreme coefficients (random AC up to +-300 and beyond) libjpeg-turbo's SIMD IDCT,
                                *    which Pillow uses by default, overflows 16-bit lanes and differs from its own C code;
                                *    this model follows the C code (JSIMD_FORCENONE=1);
                                *  - equality is claimed for 8-bit DQTs. A 16-bit DQT entry is used as parsed under the
                                *    batch's gate: without B2J_PARSE_ROBUST it is byte-swapped relative to libjpeg;
                                *  - files libjpeg would treat as RGB (Adobe transform 0, component ids 'R', 'G', 'B') are
                                *    still converted as YCbCr; in B2J_OUT_GRAY8, where libjpeg would compute luminance from
                                *    R, G and B, their first component is output as it is. */

/* reference enum ColorSpace (macro.h:114-119) */
#define B2J_CS_YUV444 0
#define B2J_CS_YUV411 1
#define B2J_CS_OTHER 2
#define B2J_CS_GRAY 3     /* not in the reference's enum: one component (B2J_GATE_GRAY) */

/* Parsed frame/scan header of one baseline JPEG: the POD equivalent of the reference's
 * JPG_DATA (jpeg.h:59-81) minus the pointers. Quantisation tables stay in file (zig-zag)
 * order like parser.cpp:65-86 keeps them; Huffman tables are kept as the DHT payload
 * (16 counts + symbols), slot = Tc*4 + Th (Tc 0 = DC, 1 = AC; Th 0..3). */
typedef struct b2j_image_desc
{
    int32_t width, height;
    uint8_t sampling[3];  /* (h<<4)|v per component, SOF0                                   */
    uint8_t quant_id[3];
    uint8_t huff_id[3];   /* (Td<<4)|Ta per component, SOS                                  */
    uint8_t color_space;  /* B2J_CS_*                                                       */
    uint8_t quant_present[4];
    uint8_t huff_present[8];
    int32_t restart_interval;
    int32_t mcu_width, mcu_height;         /* pixels                                        */
    int32_t mcu_count_w, mcu_count_h, mcu_count;
    int32_t blks_per_mcu[3];
    int32_t tot_blks_per_mcu;
    int32_t blk_count;
    uint64_t scan_offset;                  /* first entropy-coded byte                      */
    uint64_t scan_size;                    /* bytes from scan_offset to the end of the file */
    uint16_t quant[4][64];
    uint8_t huff_counts[8][16];
    uint8_t huff_symbols[8][256];
} b2j_image_desc;

typedef struct b2j_ctx b2j_ctx;
typedef struct b2j_batch b2j_batch;

/* Byte/launch accounting of one b2j_batch_decode() (for the roofline arithmetic). */
typedef struct b2j_batch_info
{
    int32_t n_images;
    int32_t kernel_launches;      /* kernels enqueued by one b2j_batch_decode()             */
    int64_t total_pixels;         /* sum W*H                                                */
    int64_t total_blocks;         /* sum blk_count (padding MCUs included)                  */
    int64_t scan_bytes;           /* sum of entropy-coded bytes uploaded                    */
    int64_t coef_plane_bytes;     /* 128 * total_blocks                                     */
    int64_t pixel_bytes;          /* 4 * total_pixels                                       */
    int64_t algorithmic_bytes;    /* scan + 2*coef_plane + pixel (SURVEY.md 8d)             */
    int64_t device_bytes;         /* device memory held by the batch                        */
    int64_t h2d_bytes;            /* bytes b2j_batch_upload() copies                        */
} b2j_batch_info;

/* Device timings of the stages of the most recent b2j_batch_decode_timed(), milliseconds. */
typedef struct b2j_stage_times
{
    float prepass_ms;   /* marker scan + unstuff + restart-interval table                   */
    float huffman_ms;   /* entropy decode -> int16 coefficient plane                        */
    float idct_ms;      /* dequant + IDCT + upsample + colour -> BGRA, and the orientation pass
                         * (b2j_batch_set_orientations) when it runs                         */
    float total_ms;
} b2j_stage_times;

/* ------------------------------------------------------------------ host-only ---------- */
int b2j_abi_version(void);
const char *b2j_strerror(int code);
/* Text of the last CUDA/runtime failure on this thread ("" when none). */
const char *b2j_last_error(void);

/* Parse SOI .. SOS of a baseline JFIF file held in memory. Same accept/reject behaviour as
 * the reference's load_jpg() + is_supported_file() (gate = B2J_GATE_REFERENCE), or with
 * 4:2:2 / 4:4:0 admitted (B2J_GATE_EXTENDED).
 * Deviation, under every gate: B2J_E_UNSUPPORTED for a file whose Huffman tables need more than 12288 entries of
 * two-level decode tables together (16 header entries, then per distinct table 64 (DC) or 1024 (AC) first-level entries
 * plus 2^(L - 6) resp. 2^(L - 10) entries for every first-level prefix whose longest code has length L, each sub-table
 * starting on a multiple of 8). The decode kernels keep them in 24 KB of shared memory. The Annex K tables need 2536
 * entries; tables with at most the 12 DC and 162 AC symbols a baseline encoder uses need at most 11656 (the largest a
 * search over code lengths finds, three components on distinct tables). Only tables of about 256 codes up to 16 bits
 * long pass the limit, e.g. three DC and two AC tables of that kind. The reference decodes such files. The check is per
 * file, so that such a file cannot make b2j_batch_create fail for the whole batch. */
int b2j_parse_header(const uint8_t *file, size_t len, int gate, b2j_image_desc *out);

/* EXIF orientation of a file held in memory: *orientation = the value of tag 0x0112 (Orientation) in IFD0 of the first
 * APP1 segment whose payload starts with "Exif\0\0" (what Pillow reads: an XMP APP1 in front of it is skipped, a second
 * Exif APP1 is not read), read as 16 bits in the TIFF header's byte order (II or MM). The length-prefixed segments from SOI
 * to SOS are walked whatever the gate. *orientation = 1 when there is no such tag, when its value is outside 1..8, and
 * when anything is cut or malformed; nothing outside [file, file + len) is read. B2J_E_ARG only for null pointers.
 * b2j_batch_set_orientations() and b2j_host_opts.exif_orientation take these codes. */
int b2j_parse_orientation(const uint8_t *file, size_t len, int32_t *orientation);

/* ------------------------------------------------------------------ device -------------- */
int b2j_device_count(void);
int b2j_create(int device, b2j_ctx **out);
void b2j_destroy(b2j_ctx *ctx);

/* Build a batch: stages the entropy-coded bytes of every image (files[i] + desc.scan_offset)
 * in pinned host memory, builds the decode tables, allocates all device buffers. Nothing is
 * copied to the device yet. */
int b2j_batch_create(b2j_ctx *ctx, int n, const b2j_image_desc *descs, const uint8_t *const *files,
                     const size_t *lens, b2j_batch **out);
void b2j_batch_destroy(b2j_batch *batch);
int b2j_batch_get_info(const b2j_batch *batch, b2j_batch_info *info);

/* stream: a cudaStream_t passed as void* (NULL = the context's own stream). All calls below
 * only enqueue work unless stated. */
int b2j_batch_upload(b2j_batch *batch, void *stream);   /* H2D: scan bytes + tables        */
int b2j_batch_decode(b2j_batch *batch, void *stream);   /* the hot path, device resident   */
/* Same as b2j_batch_decode() with CUDA events between the stages; synchronises. */
int b2j_batch_decode_timed(b2j_batch *batch, void *stream, b2j_stage_times *times);
/* `steps` decodes back to back on one stream with CUDA events recorded (not waited for) between
 * the stages of every step; synchronises once at the end. per_step: `steps` entries or NULL.
 * total_ms: first event of the first step to last event of the last step. */
int b2j_batch_decode_steps(b2j_batch *batch, void *stream, int steps, b2j_stage_times *per_step, float *total_ms);
int b2j_batch_sync(b2j_batch *batch, void *stream);

/* Layout of the pixel plane for the decodes that follow (B2J_OUT_*; default B2J_OUT_BGRA; B2J_E_ARG for an unknown one).
 * The values are the same in BGRA, RGB24 and planar RGB -- the pixel model's colour -- only their arrangement differs;
 * B2J_OUT_GRAY8 carries the luma samples instead. B2J_OUT_GRAY8 is accepted at any time, but needs B2J_PIXELS_LIBJPEG:
 * a decode in it in the reference model fails with B2J_E_ARG (b2j_last_error() says why). In the libjpeg model it runs
 * one kernel instead of two and needs no sample plane (b2j_batch_info counts both). b2j_decode_host() and the
 * reference-API shim always produce the reference's BGRA. */
int b2j_batch_set_output_format(b2j_batch *batch, int format);
/* Pixel model for the decodes that follow (B2J_PIXELS_*; default B2J_PIXELS_REFERENCE), with every output format and
 * with b2j_batch_downscale(). The coefficients and the status words are the same in both models; only the stage after
 * the coefficient plane differs. B2J_PIXELS_LIBJPEG runs two kernels instead of one per tile kind, and the first decode
 * in it in a format other than B2J_OUT_GRAY8 allocates a sample plane of 64 bytes per block (b2j_batch_info counts
 * both). B2J_E_ARG for an unknown model. */
int b2j_batch_set_pixel_model(b2j_batch *batch, int model);
/* Scale of the decodes that follow: denom 1 (default), 2, 4 or 8, B2J_E_ARG for any other value. Reduced size:
 * ceil(w/denom) x ceil(h/denom), in the batch's output format, at the image's usual place with tight pitch (the reads,
 * b2j_batch_pixels_device and the host calls follow it). This is libjpeg-turbo's scaled decode (scale_num = 1,
 * scale_denom = denom; Pillow's Image.draft()): the reduced IDCTs of jidctred.c, each component at the DCT size
 * jdmaster.c chooses, then jdsample.c's upsampling (no fancy filter at 1/8) and the same colour conversion. It needs
 * B2J_PIXELS_LIBJPEG: a decode with denom != 1 in the reference model fails with B2J_E_ARG (b2j_last_error() says why),
 * and so does b2j_batch_downscale() while denom != 1. The coefficients, the status words and b2j_batch_info do not
 * change; the sample plane keeps its size. */
int b2j_batch_set_scale(b2j_batch *batch, int denom);
/* EXIF orientation of every image for the decodes that follow: codes[i] in 1..8 (b2j_parse_orientation), NULL = 1 for
 * every image (the default); B2J_E_ARG for any other code, and then nothing changes. An image of w x h pixels at the
 * batch's scale is decoded as before, then transformed (numpy, a = the (h, w, ...) image): 1 a, 2 a[:, ::-1],
 * 3 a[::-1, ::-1], 4 a[::-1], 5 a.swapaxes(0, 1), 6 a.swapaxes(0, 1)[:, ::-1], 7 a.swapaxes(0, 1)[::-1, ::-1],
 * 8 a.swapaxes(0, 1)[::-1]; codes 5..8 give h x w pixels. Planar RGB: each plane. Scaled decode first, then orientation:
 * what OpenCV's cv2.imdecode / cv2.imread give with their default flags (IMREAD_COLOR, IMREAD_GRAYSCALE,
 * IMREAD_REDUCED_*; only IMREAD_IGNORE_ORIENTATION turns it off), torchvision's decode_jpeg(..., apply_exif_orientation=True)
 * and Pillow's ImageOps.exif_transpose(). In both pixel models, every output format and every scale. The oriented
 * pixels have tight pitch in the batch's format and as many bytes as the unoriented ones; b2j_batch_pixels_device and
 * the reads return them. One more kernel runs after the IDCT/colour stage over the images whose code is not 1, into a
 * buffer of their own (b2j_batch_info counts both); with every code 1 a decode is what it is without this call.
 * b2j_batch_downscale() is refused (B2J_E_ARG) while a code is not 1. */
int b2j_batch_set_orientations(b2j_batch *batch, const uint8_t *codes /* n or NULL */);
/* A crop box per image for the decodes that follow: boxes[4*i .. 4*i+3] = x, y, w, h of image i, NULL = the whole images
 * (the default); B2J_E_ARG for a negative value or w or h < 1, and then nothing changes. A box is given in the frame the
 * decode would otherwise deliver: the image at the batch's scale (b2j_batch_set_scale), then oriented by its code
 * (b2j_batch_set_orientations; codes 5..8 swap the sides). The result is exactly that image's [y:y+h, x:x+w] (numpy;
 * planar RGB: each plane), w x h pixels with tight pitch in the batch's format, in every format and at every scale:
 * Pillow's draft(), exif_transpose(), then crop((x, y, x+w, y+h)); torchvision's decode_jpeg(..., apply_exif_orientation=
 * True)[..., y:y+h, x:x+w]. b2j_batch_pixels_device and the reads return it. The box is checked at each decode, since the
 * scale and the codes may change after this call: a box that does not lie inside its frame fails the decode, and the
 * reads, with B2J_E_ARG, and b2j_last_error() names the image. Needs B2J_PIXELS_LIBJPEG: a decode with crops in the
 * reference model fails with B2J_E_ARG. b2j_batch_downscale() is refused (B2J_E_ARG) while crops are set.
 * Only the MCUs the window touches, with one MCU around them for fancy upsampling (none in GRAY8 and at scale 8), are
 * transformed, and only the window is upsampled and coloured; the pre-pass and the entropy stage decode the whole scan,
 * so the status words and the coefficients are those of the uncropped decode. The windows and their tile list live in a
 * buffer of their own (b2j_batch_info counts it); with NULL a decode is what it is without this call. */
int b2j_batch_set_crops(b2j_batch *batch, const int32_t *boxes /* 4*n or NULL */);

/* Per-image status words (B2J_ST_* bits). Synchronises the stream. */
int b2j_batch_status(b2j_batch *batch, void *stream, int32_t *status /* n */);

/* Convergence evidence of the self-synchronising entropy decoder (streams without DRI) for the most
 * recent decode: out8[r] = sub-sequence exit states that round r (1..) still changed, out8[7] =
 * sub-sequences the sequential sweep had to re-walk. Synchronises. */
int b2j_batch_sync_stats(b2j_batch *batch, void *stream, uint32_t *out8);

/* Device-resident results. Pixels: top-down, tight pitch, in the batch's output format (BGRA: width*4 per row, A = 0),
 * at the batch's scale (b2j_batch_set_scale: width and height are then the reduced ones), oriented, cropped
 * (b2j_batch_set_crops: w x h). */
int b2j_batch_pixels_device(const b2j_batch *batch, int image, void **dptr, size_t *nbytes);
/* Coefficient plane: int16[blk_count][64], natural order, QUANTISED (dequantisation happens
 * at IDCT load), MCU-interleaved block order. */
int b2j_batch_coefs_device(const b2j_batch *batch, int image, void **dptr, size_t *nbytes);

/* D2H of one image (synchronises). dst: width*height*4 bytes (BGRA), width*height*3 (RGB24, planar RGB) or width*height
 * (GRAY8), of the size at the batch's scale, oriented; a crop box's w*h pixels with crops. */
int b2j_batch_read_pixels(b2j_batch *batch, void *stream, int image, uint8_t *dst);
/* D2H of every image into dsts[i] (pinned staging, one copy per image; synchronises). */
int b2j_batch_read_all_pixels(b2j_batch *batch, void *stream, uint8_t *const *dsts);
/* The reference's coefficient tap: int32[blk_count][64], natural order, dequantised on the
 * device by a small expansion kernel, then copied (synchronises). */
int b2j_batch_read_coefs(b2j_batch *batch, void *stream, int image, int32_t *dst);

/* Output stage for consumers that want smaller images (SURVEY.md 8f rank 3): box-filter reduction of the decoded pixels by
 * factor 2, 4 or 8 per axis, after b2j_batch_decode(), in the batch's output format. Reduced size: ceil(w/f) x ceil(h/f);
 * every value is the rounded mean (sum + n/2) / n of the n input values it covers (at the right / bottom edge: of those that
 * exist). The full-size pixels stay where they are. B2J_E_ARG while the batch's scale (b2j_batch_set_scale) is not 1,
 * while an orientation code (b2j_batch_set_orientations) is not 1, and while crops (b2j_batch_set_crops) are set. */
int b2j_batch_downscale(b2j_batch *batch, void *stream, int factor);
int b2j_batch_downscaled_device(const b2j_batch *batch, int image, void **dptr, size_t *nbytes, int *width, int *height);
int b2j_batch_read_downscaled(b2j_batch *batch, void *stream, int image, uint8_t *dst);   /* synchronises */

/* Whole path with host buffers in and out: parse, upload, decode, download.
 * out_bgra[i] must hold width*height*4 bytes (use b2j_parse_header() to size it); images whose
 * header is rejected get status[i] = the negative B2J_E_* code and are skipped. */
int b2j_decode_host(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, int gate,
                    uint8_t *const *out_bgra, int32_t *status);

/* Options of b2j_decode_host_ex() / b2j_decode_host_multi(); zero-initialise, then set what differs. */
typedef struct b2j_host_opts
{
    int32_t gate;        /* B2J_GATE_* and the OR-able parse flags                                                */
    int32_t out_format;  /* B2J_OUT_*: BGRA (w*h*4 bytes per image), RGB24 or planar RGB (w*h*3 bytes), GRAY8 (w*h)  */
    int32_t n_threads;   /* host threads that parse headers and stage scans into pinned memory; 0 = as many as
                          * the machine offers, at most 8                                                        */
    int32_t group;       /* images per pipeline group (0 = 32): a group is uploaded, decoded and read back as one */
    int32_t group_mb;    /* and at most this many MiB of files per group (0 = 12): one host thread stages a group  */
    int32_t pixel_model; /* B2J_PIXELS_* (0 = the reference's pixels)                                             */
    int32_t scale;       /* 1, 2, 4 or 8 (0 = 1): b2j_batch_set_scale(); needs B2J_PIXELS_LIBJPEG                     */
    int32_t exif_orientation; /* 0: as decoded; 1: each file's b2j_parse_orientation() code applied
                               * (b2j_batch_set_orientations()), so out[i] holds the oriented image, sides swapped for 5..8 */
} b2j_host_opts;

/* b2j_decode_host() with options: the pixels arrive in opts->out_format (RGB24 moves 25 % fewer bytes over PCIe,
 * which is what bounds this call) and opts->pixel_model (B2J_E_ARG for an unknown one), headers are parsed and scans
 * staged by opts->n_threads host threads while the calling thread only enqueues uploads, decodes and downloads.
 * out[i]: w*h*4, w*h*3 or w*h (GRAY8) bytes, with w = ceil(width/scale) and h = ceil(height/scale) for opts->scale
 * (B2J_E_ARG for a scale other than 0, 1, 2, 4 and 8, and for a scale other than 1 or B2J_OUT_GRAY8 in the reference
 * pixel model). With opts->exif_orientation = 1 (B2J_E_ARG for a value other than 0 and 1) out[i] holds the image
 * oriented by its EXIF code: h*w bytes per channel with the sides swapped for codes 5..8. b2j_decode_host() does not
 * orient. b2j_decode_host_ex() is b2j_decode_host_crop() with crops = NULL. */
int b2j_decode_host_ex(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, const b2j_host_opts *opts,
                       uint8_t *const *out, int32_t *status);
/* b2j_decode_host_ex() with a crop box per file (crops[4*i .. 4*i+3] = x, y, w, h; NULL = none), as
 * b2j_batch_set_crops() takes it: in the file's frame at opts->scale, oriented when opts->exif_orientation = 1.
 * out[i] holds the box's w*h pixels (w*h*4, w*h*3 or w*h bytes). A file whose box does not lie inside its frame (a
 * negative value, w or h < 1 included) gets status[i] = B2J_E_ARG and is skipped; the others are decoded. Needs
 * B2J_PIXELS_LIBJPEG when crops is not NULL (B2J_E_ARG for the whole call otherwise). */
int b2j_decode_host_crop(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, const b2j_host_opts *opts,
                         const int32_t *crops /* 4*n or NULL */, uint8_t *const *out, int32_t *status);

/* The same over several devices: ctxs[k] = a context on the k-th device to use (b2j_create(device)); image i goes to
 * exactly one of them (contiguous index ranges of about equal compressed size). One host thread per context runs
 * b2j_decode_host_ex() on its range; nothing is exchanged between devices. Returns the first failure, if any. */
int b2j_decode_host_multi(b2j_ctx *const *ctxs, int n_ctx, int n, const uint8_t *const *files, const size_t *lens,
                          const b2j_host_opts *opts, uint8_t *const *out, int32_t *status);

/* Pinned (page-locked, all devices) host memory for inputs and outputs of the calls above. */
int b2j_host_alloc(void **out, size_t bytes);
void b2j_host_free(void *p);

/* Reads n whole files with n_threads (0 = auto) into one pinned arena: files[i] / lens[i] are filled in, *arena is
 * what to pass to b2j_host_free() afterwards. A file that cannot be read gets files[i] = NULL, lens[i] = 0 and the
 * call returns B2J_E_ARG after reading the others. */
int b2j_read_files(int n, const char *const *paths, int n_threads, void **arena, const uint8_t **files, size_t *lens);

/* ------------------------------------------------------------------ secondary boundary -- */
/* Coefficients in, pixels out: the reference's device backend (idct.h:9-18, oclDCT8x8.cpp) as it is driven by the
 * reference's own decoder.cpp, which entropy-decodes on the CPU and hands over int32 coefficients that are already
 * dequantised. csrc/refshim/idct_b2j.cpp implements the ten clidct_* functions on these calls.
 *   b2j_idct_create        clidct_create() + clidct_allocate_memory() + clidct_build()   (idct.h:10-11,13)
 *   b2j_idct_upload        clidct_transfer_data_to_device()                              (idct.h:12)
 *   b2j_idct_run           clidct_run() + clidct_wait_for_completion()                   (idct.h:14,17)
 *   b2j_idct_read_pixels   clidct_retrieve_image_from_device()                           (idct.h:16)
 *   b2j_idct_read_coefs    clidct_retrieve_data_from_device()                            (idct.h:15)
 *   b2j_idct_destroy       clidct_clean_up()                                             (idct.h:18)
 * Luma sampling luma_h x luma_v with 1x1 chroma: the reference's YUV444 is (1,1), its YUV411 (2,2). The coefficients are
 * int32 [blk_count][64], natural order, MCU-interleaved block order (JPG_DATA::mcu_data, jpeg.h:74); they are held as
 * int16 on the device (saturated; an 8-bit baseline JPEG keeps them inside +-2^15). The pixels equal the reference's CPU
 * path (cpuIDCT8x8 + YUV_to_RGB32), not the OpenCL kernel's float colour. */
typedef struct b2j_idct b2j_idct;
int b2j_idct_create(b2j_ctx *ctx, int width, int height, int luma_h, int luma_v, b2j_idct **out);
int b2j_idct_blk_count(const b2j_idct *p);
int b2j_idct_upload(b2j_idct *p, const int32_t *coefs, int offset, int count);
int b2j_idct_run(b2j_idct *p);
int b2j_idct_read_pixels(b2j_idct *p, uint8_t *bgra /* width*height*4 */);
int b2j_idct_read_coefs(b2j_idct *p, int32_t *coefs /* blk_count*64 */);
void b2j_idct_destroy(b2j_idct *p);

#ifdef __cplusplus
}
#endif
#endif /* B2J_H_INCLUDED */
