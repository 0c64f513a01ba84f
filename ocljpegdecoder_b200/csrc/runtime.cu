// runtime.cu -- the extern "C" layer: contexts, batches, uploads, launches, read-back.
//
// Replaces the reference's OpenCL host runtime (oclDCT8x8.cpp:25-341: device discovery,
// context/queue, buffers, blocking transfers, run-time program build, launch, teardown) with a
// CUDA runtime layer in which whole batches of images stay resident on one B200:
//   b2j_batch_create   lays out every buffer of a batch once (compressed scans, tables, segment
//                      and tile descriptors, coefficient plane, pixel plane)
//   b2j_batch_upload   one host->device copy of the packed input blob
//   b2j_batch_decode   the pre-pass, entropy and IDCT/colour kernels in order on one stream, no host
//                      synchronisation
// There is no CPU fallback anywhere in this file: without a device every call fails.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <map>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "b2j_internal.h"
#include "b2j_math.h"
#include "crop_plan.h"
#include "kernels.h"

using namespace b2j;

namespace {

thread_local std::string t_last_error;

int fail_cuda(cudaError_t e, const char *what)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    t_last_error = buf;
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? B2J_E_NODEVICE : B2J_E_CUDA;
}

#define CU_TRY(expr)                                              \
    do {                                                          \
        cudaError_t e__ = (expr);                                 \
        if (e__ != cudaSuccess) return fail_cuda(e__, #expr);     \
    } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// A buffer held from a Pool; empty (null, capacity 0) when none is held.
struct PoolBuf
{
    void *p = nullptr;
    size_t cap = 0;
};

// A grow-only cache of device / pinned allocations so that repeated batches (the e2e path) do
// not pay cudaMalloc / cudaHostAlloc every call.
struct Pool
{
    std::vector<PoolBuf> free_list;
    bool pinned;
    explicit Pool(bool pin) : pinned(pin) {}
    // fills the empty `b` with at least n bytes; leaves it empty on failure
    cudaError_t get(size_t n, PoolBuf &b)
    {
        size_t best = (size_t)-1;
        for (size_t i = 0; i < free_list.size(); i++)
            if (free_list[i].cap >= n && (best == (size_t)-1 || free_list[i].cap < free_list[best].cap)) best = i;
        if (best != (size_t)-1)
        {
            b = free_list[best];
            free_list.erase(free_list.begin() + (long)best);
            return cudaSuccess;
        }
        n = align_up(n ? n : 1, 1 << 20);
        void *p = nullptr;
        const cudaError_t e = pinned ? cudaHostAlloc(&p, n, cudaHostAllocDefault) : cudaMalloc(&p, n);
        if (e == cudaSuccess) b = {p, n};
        return e;
    }
    // hands `b` back and leaves it empty
    void put(PoolBuf &b)
    {
        if (b.p) free_list.push_back(b);
        b = {};
    }
    void drain()
    {
        for (auto &b : free_list) { if (pinned) cudaFreeHost(b.p); else cudaFree(b.p); }
        free_list.clear();
    }
};

} // namespace

struct b2j_ctx
{
    int device;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;   // host feed: the downloads of a group run here while the next group decodes on `stream`
    PFN_cuTensorMapEncodeTiled_v12000 encode_tiled;
    int sm_count;
    Pool dev_pool{false};
    Pool pin_pool{true};
    std::mutex mu;
};

struct b2j_batch
{
    b2j_ctx *ctx;
    int n;
    std::vector<ImgDev> imgs;
    b2j_batch_info info;

    // packed input blob: host (pinned) and device copies share one layout
    PoolBuf h_blob, d_blob;
    size_t blob_bytes;
    ImgDev *h_imgs;      // the image table in the pinned blob

    // scratch + outputs; the DecodeArgs pointers lead into them
    PoolBuf d_scratch, d_coef, d_pix;
    size_t clean_bytes;  // the clean stream and its tail, from args.clean: defined by the first upload
    size_t zero_bytes;   // the status words, sync stats and look-back words, from args.status: zeroed by every decode
    size_t coef_rows;
    uint32_t n_segs_total;
    PoolBuf d_expand;    // lazily allocated for the coefficient tap
    PoolBuf d_small;     // lazily allocated: the reduced pixels of b2j_batch_downscale() behind a table of offsets
    PoolBuf d_samples;   // lazily allocated by the first decode in the libjpeg pixel model: its sample plane
    int small_factor = 0;                     // 0 = none
    std::vector<uint64_t> small_off;          // byte offset of every image's reduced pixels behind the offset table
    // EXIF orientation (b2j_batch_set_orientations): d_orient holds the orientation pass's tile table, then the oriented
    // copies of the images whose code is not 1, in image order; h_orient is the pinned staging of the table
    std::vector<uint8_t> orient;              // one code per image; empty = every code 1
    std::vector<uint64_t> orient_off;         // byte offset of an oriented image's copy in d_orient
    PoolBuf d_orient, h_orient;
    size_t orient_table_bytes = 0;            // room for the table at scale 1, where an image has the most tiles
    uint32_t n_orient_tiles = 0;
    bool orient_stale = false;                // the table on the device is not the one of the current settings
    cudaEvent_t orient_copied = nullptr;      // the last copy out of h_orient
    // crop windows (b2j_batch_set_crops): d_crop holds every image's window, the window views that the orientation pass
    // reads as its image table (an image the size of its window), then the crop tile list; h_crop is their pinned staging
    std::vector<int32_t> crops;               // x, y, w, h per image, in the oriented frame at the batch's scale; empty = none
    std::vector<CropDev> win;                 // every image's window in its unoriented frame (set_output)
    int crop_misfit = -1;                     // the first image whose box does not fit its frame (set_output); -1 = none
    PoolBuf d_crop, h_crop;
    size_t crop_views_off = 0, crop_tiles_off = 0;
    bool crop_stale = false;                  // the windows and tiles on the device are not those of the current settings
    cudaEvent_t crop_copied = nullptr;        // the last copy out of h_crop

    CUtensorMap tmap;
    DecodeArgs args;
    int fixed_launches;   // the kernels of a decode before the IDCT/colour stage: pre-pass and entropy stage
    bool uploaded = false;
    cudaStream_t last_stream = nullptr;   // the stream the batch was last uploaded / decoded / read on
};

namespace {

int make_tensor_map(b2j_ctx *ctx, b2j_batch *b)
{
    memset(&b->tmap, 0, sizeof(b->tmap));
    // coefficient plane as a 2-D tensor [rows][64] of int16; box = one tile, 128-byte swizzle
    const cuuint64_t dims[2] = {64, (cuuint64_t)b->coef_rows};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {64, (cuuint32_t)kTileBlocks};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = ctx->encode_tiled(&b->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, b->d_coef.p, dims, strides, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
    {
        char buf[128];
        snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed: CUresult %d", (int)r);
        t_last_error = buf;
        return B2J_E_CUDA;
    }
    return B2J_OK;
}

uint32_t mode_of(const b2j_image_desc &d)
{
    if (d.color_space == B2J_CS_GRAY) return kModeGray;
    if (d.sampling[1] != 0x11 || d.sampling[2] != 0x11) return kModeGeneric;
    switch (d.sampling[0])
    {
    case 0x11: return kMode444;
    case 0x22: return kMode420;
    case 0x21: return kMode422;
    case 0x12: return kMode440;
    default: return kModeGeneric;
    }
}

// The descriptor is caller-supplied: every derived field is recomputed from width, height and the sampling
// factors (decoder.cpp:161-192) and must agree, so that no kernel ever indexes with an inconsistent geometry.
bool geometry_ok(const b2j_image_desc &d)
{
    if (d.width <= 0 || d.height <= 0 || d.width > 65535 || d.height > 65535) return false;
    const bool gray = d.color_space == B2J_CS_GRAY;
    int mh = 0, mv = 0, tot = 0, blks[3] = {0, 0, 0};
    for (int c = 0; c < (gray ? 1 : 3); c++)
    {
        const int h = d.sampling[c] >> 4, v = d.sampling[c] & 0xF;
        if (h < 1 || h > 4 || v < 1 || v > 4) return false;
        mh = h > mh ? h : mh; mv = v > mv ? v : mv;
        blks[c] = h * v; tot += h * v;
    }
    if (tot > 10) return false;
    // the kernels replicate chroma samples: the chroma factors must divide the luma's (what the gate admits)
    for (int c = 1; c < (gray ? 1 : 3); c++)
        if ((d.sampling[0] >> 4) % (d.sampling[c] >> 4) || (d.sampling[0] & 0xF) % (d.sampling[c] & 0xF)) return false;
    const int mcw = (d.width - 1) / (8 * mh) + 1, mch = (d.height - 1) / (8 * mv) + 1;
    if (d.mcu_width != 8 * mh || d.mcu_height != 8 * mv || d.mcu_count_w != mcw || d.mcu_count_h != mch) return false;
    if (d.mcu_count != mcw * mch || d.tot_blks_per_mcu != tot || d.blk_count != d.mcu_count * tot) return false;
    for (int c = 0; c < 3; c++)
        if (d.blks_per_mcu[c] != blks[c] || d.quant_id[c] > 3) return false;
    if (d.restart_interval < 0) return false;
    return true;
}

cudaStream_t pick_stream(b2j_batch *b, void *stream) { return b->last_stream = (stream ? (cudaStream_t)stream : b->ctx->stream); }

// Grows the device (or, `pinned`, page-locked host) buffer `buf` to at least n bytes from the context's pool; its contents
// are not kept. On failure the buffer is left empty and CUDA's last error is cleared, so that it cannot fail the next,
// unrelated call on this thread.
cudaError_t grow(b2j_ctx *ctx, PoolBuf &buf, size_t n, bool pinned = false)
{
    if (buf.cap >= n) return cudaSuccess;
    std::lock_guard<std::mutex> lk(ctx->mu);
    Pool &pool = pinned ? ctx->pin_pool : ctx->dev_pool;
    pool.put(buf);
    const cudaError_t e = pool.get(n, buf);
    if (e != cudaSuccess) cudaGetLastError();
    return e;
}

template <class T> T *at(const PoolBuf &buf, size_t off) { return reinterpret_cast<T *>((uint8_t *)buf.p + off); }

void release_orient_buffers(b2j_batch *b)
{
    b2j_ctx *c = b->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    c->dev_pool.put(b->d_orient);
    c->pin_pool.put(b->h_orient);
}

void release_crop_buffers(b2j_batch *b)
{
    b2j_ctx *c = b->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    c->dev_pool.put(b->d_crop);
    c->pin_pool.put(b->h_crop);
}

void release_batch_buffers(b2j_batch *b)
{
    release_orient_buffers(b);
    release_crop_buffers(b);
    for (cudaEvent_t *e : {&b->orient_copied, &b->crop_copied})
    {
        if (*e) cudaEventDestroy(*e);
        *e = nullptr;
    }
    b2j_ctx *c = b->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    c->pin_pool.put(b->h_blob);
    for (PoolBuf *d : {&b->d_blob, &b->d_scratch, &b->d_coef, &b->d_pix, &b->d_expand, &b->d_small, &b->d_samples}) c->dev_pool.put(*d);
}

// b2j_batch_info::device_bytes: the buffers a decode uses (the read-back buffers of the coefficient tap and of
// b2j_batch_downscale() are not counted)
int64_t device_bytes(const b2j_batch *b)
{
    return (int64_t)(b->d_blob.cap + b->d_scratch.cap + b->d_coef.cap + b->d_pix.cap + b->d_samples.cap + b->d_orient.cap + b->d_crop.cap);
}

// The image `image` of the batch, or nullptr when the batch has no such image.
const ImgDev *image_of(const b2j_batch *b, int image) { return b && image >= 0 && image < b->n ? &b->imgs[(size_t)image] : nullptr; }

// Bytes per pixel of an output format (B2J_OUT_*).
size_t format_bpp(int fmt) { return fmt == B2J_OUT_BGRA ? 4 : (fmt == B2J_OUT_GRAY8 ? 1 : 3); }

bool format_ok(int fmt) { return fmt == B2J_OUT_BGRA || fmt == B2J_OUT_RGB24 || fmt == B2J_OUT_RGB_PLANAR || fmt == B2J_OUT_GRAY8; }

bool model_ok(int model) { return model == B2J_PIXELS_REFERENCE || model == B2J_PIXELS_LIBJPEG; }

bool scale_ok(int denom) { return denom == 1 || denom == 2 || denom == 4 || denom == 8; }

// Why a decode with these settings cannot run, or nullptr when it can. The setters store any valid value, so a batch
// may hold such a combination; the decode refuses it.
const char *output_refusal(int model, int fmt, int scale, bool cropped)
{
    if (model == B2J_PIXELS_LIBJPEG) return nullptr;
    if (scale != 1) return "a scaled decode (b2j_batch_set_scale, b2j_host_opts.scale) needs the libjpeg pixel model: the reference has none";
    if (fmt == B2J_OUT_GRAY8) return "B2J_OUT_GRAY8 (libjpeg's grayscale output) needs the libjpeg pixel model: the reference has none";
    if (cropped) return "a cropped decode (b2j_batch_set_crops, b2j_decode_host_crop) needs the libjpeg pixel model";
    return nullptr;
}

// An image's size with each side divided by `div`, rounded up: the output of a decode at scale `div`, or the reduced
// copy of b2j_batch_downscale() by factor `div`.
struct Dims { uint32_t w, h; };
Dims out_dims(const ImgDev &im, uint32_t div) { return {(im.width + div - 1) / div, (im.height + div - 1) / div}; }

// What a decode delivers of image i: scale, then crop, then orientation. `win` is the window the IDCT/colour stage
// writes, in the image's unoriented frame at the batch's scale (the whole frame without crops); `dims` is the size of the
// result the reads return (the window, sides swapped for orientation codes 5..8).
struct ImageOut { CropDev win; Dims dims; };
ImageOut image_out(const b2j_batch *b, size_t i)
{
    const Dims f = out_dims(b->imgs[i], b->args.scale);
    const CropDev win = b->crops.empty() ? CropDev{0, 0, f.w, f.h} : b->win[i];
    const bool swap = !b->orient.empty() && b->orient[i] >= 5;
    return {win, swap ? Dims{win.h, win.w} : Dims{win.w, win.h}};
}

size_t image_bytes(const b2j_batch *b, size_t i)
{
    const Dims o = image_out(b, i).dims;
    return (size_t)o.w * o.h * format_bpp(b->args.out_format);
}

// B2J_E_ARG, naming the image, while a crop box does not lie inside its image's frame at the batch's scale and orientation.
int crop_refusal(const b2j_batch *b)
{
    if (b->crop_misfit < 0) return B2J_OK;
    const ImgDev &im = b->imgs[(size_t)b->crop_misfit];
    const Dims f = out_dims(im, b->args.scale);
    const bool swap = !b->orient.empty() && b->orient[(size_t)b->crop_misfit] >= 5;
    const int32_t *c = &b->crops[4 * (size_t)b->crop_misfit];
    char buf[256];
    snprintf(buf, sizeof(buf), "the crop box (%d, %d, %d, %d) of image %d does not lie inside its %u x %u frame (at the batch's scale, oriented)", c[0], c[1],
             c[2], c[3], b->crop_misfit, swap ? f.h : f.w, swap ? f.w : f.h);
    t_last_error = buf;
    return B2J_E_ARG;
}

// Alignment of an image's start when images are packed side by side in a format: what the stores of the kernels that
// write them allow (16 bytes for BGRA, 4 for the three-byte formats, none for GRAY8, whose kernels store single bytes).
size_t pack_align(int fmt) { return fmt == B2J_OUT_BGRA ? 16 : (fmt == B2J_OUT_GRAY8 ? 1 : 4); }

// The only writer of a batch's output settings and of what follows from them: the crop windows, the upsampling kernel's
// grid, the places of the oriented copies and the launch count of a decode.
void set_output(b2j_batch *b, int model, int fmt, int scale)
{
    b->args.pixel_model = model;   // the sample plane, once allocated, stays with the batch
    b->args.out_format = fmt;      // the pixel plane is sized for BGRA at scale 1: every format, scale and crop fits
    b->args.scale = (uint32_t)scale;
    // the windows of the crop boxes; a box that does not fit the frame stands for the whole frame until the settings
    // change, and decodes and reads are refused (crop_refusal)
    b->crop_misfit = -1;
    for (size_t i = 0; i < b->crops.size() / 4; i++)
    {
        const Dims f = out_dims(b->imgs[i], (uint32_t)scale);
        if (!crop_window(f.w, f.h, b->orient.empty() ? 1u : b->orient[i], &b->crops[4 * i], b->win[i]))
        {
            b->win[i] = {0, 0, f.w, f.h};
            if (b->crop_misfit < 0) b->crop_misfit = (int)i;
        }
    }
    b->crop_stale = !b->crops.empty();
    b->args.crops = b->crops.empty() ? nullptr : at<const CropDev>(b->d_crop, 0);
    b->args.crop_tiles = b->crops.empty() ? nullptr : at<const TileDev>(b->d_crop, b->crop_tiles_off);
    uint32_t groups = 0;           // one thread per 4 output pixels of a row
    for (size_t i = 0; i < b->imgs.size(); i++)
    {
        const CropDev w = image_out(b, i).win;
        groups = std::max(groups, (w.w + 3) / 4 * w.h);
    }
    b->args.max_px_groups = groups;
    // the oriented copies behind the tile table, neighbours in image order (d_orient is sized for BGRA at scale 1); the
    // table itself follows the settings at the next decode
    size_t off = b->orient_table_bytes;
    for (size_t i = 0; i < b->orient.size(); i++)
        if (b->orient[i] != 1)
        {
            b->orient_off[i] = off = align_up(off, pack_align(fmt));
            off += image_bytes(b, i);
        }
    b->orient_stale = !b->orient.empty();
    b->info.kernel_launches = b->fixed_launches + idct_launches(b->args) + (b->orient.empty() ? 0 : 1);
}

// One device->host copy on the call's stream, waited for.
int read_back(b2j_batch *b, void *stream, void *dst, const void *src, size_t bytes)
{
    CU_TRY(cudaSetDevice(b->ctx->device));
    const cudaStream_t s = pick_stream(b, stream);
    CU_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    return B2J_OK;
}

// Copies a host-built array to its place in the pinned blob; returns where it lands on the device.
template <class T> const T *stage(const b2j_batch *b, size_t off, const std::vector<T> &v)
{
    memcpy(at<T>(b->h_blob, off), v.data(), sizeof(T) * v.size());
    return at<const T>(b->d_blob, off);
}

// Where image i's pixels are read from: its oriented copy when its orientation code is not 1, else the pixel plane.
uint8_t *result_of(const b2j_batch *b, size_t i)
{
    if (!b->orient.empty() && b->orient[i] != 1) return at<uint8_t>(b->d_orient, b->orient_off[i]);
    return b->args.pixels + b->imgs[i].pix_off;
}

} // namespace

// ---------------------------------------------------------------------------------------
extern "C" int b2j_abi_version(void) { return B2J_ABI_VERSION; }

extern "C" const char *b2j_strerror(int code)
{
    switch (code)
    {
    case B2J_OK: return "ok";
    case B2J_E_ARG: return "bad argument";
    case B2J_E_FORMAT: return "malformed or unsupported container";
    case B2J_E_UNSUPPORTED: return "rejected by the accept gate";
    case B2J_E_DATA: return "corrupt entropy-coded data";
    case B2J_E_NOMEM: return "out of memory";
    case B2J_E_CUDA: return "CUDA failure";
    case B2J_E_NODEVICE: return "no usable CUDA device (there is no CPU fallback)";
    default: return "unknown";
    }
}

extern "C" const char *b2j_last_error(void) { return t_last_error.c_str(); }

extern "C" int b2j_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int b2j_create(int device, b2j_ctx **out)
{
    if (!out) return B2J_E_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
    {
        cudaGetLastError();
        t_last_error = "no CUDA device visible; this library has no CPU fallback";
        return B2J_E_NODEVICE;
    }
    if (device < 0 || device >= n) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
    {
        t_last_error = std::string("device ") + prop.name + " is not sm_100-class; kernels are built for sm_100a only";
        return B2J_E_NODEVICE;
    }
    // the colour kernel loads its tiles through a tensor map
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
    {
        cudaGetLastError();
        t_last_error = "the driver does not export cuTensorMapEncodeTiled (needed for the TMA tile loads)";
        return B2J_E_CUDA;
    }
    b2j_ctx *ctx = new b2j_ctx;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->encode_tiled = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    cudaError_t ce = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = init_constants();
    if (ce == cudaSuccess) ce = configure_kernels(kLutMaxEntries);
    if (ce != cudaSuccess)
    {
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
        delete ctx;
        return fail_cuda(ce, "b2j_create");
    }
    *out = ctx;
    return B2J_OK;
}

extern "C" void b2j_destroy(b2j_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->dev_pool.drain();
    ctx->pin_pool.drain();
    cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->stream2);
    delete ctx;
}

// coef_only: a batch for the secondary boundary (b2j_idct_*): no scan, no decode tables, unit quantisers -- the
// coefficient plane is filled from outside, only launch_idct() runs on it.
static int batch_create_impl(b2j_ctx *ctx, int n, const b2j_image_desc *descs, const uint8_t *const *files,
                             const size_t *lens, bool coef_only, b2j_batch **out);

extern "C" int b2j_batch_create(b2j_ctx *ctx, int n, const b2j_image_desc *descs, const uint8_t *const *files,
                                const size_t *lens, b2j_batch **out)
{
    if (!files || !lens) return B2J_E_ARG;
    return batch_create_impl(ctx, n, descs, files, lens, false, out);
}

static int batch_create_impl(b2j_ctx *ctx, int n, const b2j_image_desc *descs, const uint8_t *const *files,
                             const size_t *lens, bool coef_only, b2j_batch **out)
{
    if (!ctx || n <= 0 || !descs || !out) return B2J_E_ARG;
    *out = nullptr;
    CU_TRY(cudaSetDevice(ctx->device));

    b2j_batch *b = new b2j_batch();
    b->ctx = ctx;
    b->n = n;
    b->imgs.resize((size_t)n);

    std::vector<uint32_t> chunk_img;
    std::vector<HuffCtaDev> ctas;    // restart-interval path
    std::vector<HuffCtaDev> sctas;   // self-synchronising path (no DRI)
    std::vector<uint32_t> simgs;
    uint32_t sub_total = 0;
    std::vector<TileDev> tiles;
    std::vector<uint16_t> luts;
    std::vector<uint16_t> qtabs((size_t)n * 192);
    struct LutRef { uint32_t off, len, dec_len; };
    std::map<std::string, LutRef> lut_cache;
    static const uint8_t zz[64] = B2J_ZIGZAG_TABLE;

    size_t raw_total = 0, pix_total = 0, blk_total = 0;
    uint32_t seg_total = 0, max_lut_len = 0, max_lut_dec_len = 0, max_lut_walk_len = 0;
    int64_t pixels = 0, scan_bytes = 0;
    int rc = B2J_OK;
    for (int i = 0; i < n && rc == B2J_OK; i++)
    {
        const b2j_image_desc &d = descs[i];
        ImgDev &im = b->imgs[(size_t)i];
        memset(&im, 0, sizeof(im));
        // bit positions are 32-bit on the device (scan_size * 8 must fit); an empty scan (file cut right behind the SOS
        // header) has nothing to decode -- the reference fails it with "data incomplete" (decoder.cpp:310-314)
        if (coef_only) { if (!geometry_ok(d)) { rc = B2J_E_ARG; break; } }
        else if (d.scan_offset > lens[i] || d.scan_size > lens[i] - d.scan_offset || d.scan_size == 0 || d.scan_size >= 0x1FFFFFFFull || !geometry_ok(d))
        { rc = d.scan_size == 0 && d.scan_offset <= lens[i] ? B2J_E_DATA : B2J_E_ARG; break; }
        im.raw_off = raw_total;
        im.raw_len = coef_only ? 0u : (uint32_t)d.scan_size;
        raw_total += align_up((size_t)im.raw_len + 32, 16);
        im.pix_off = pix_total;
        pix_total += align_up((size_t)d.width * d.height * 4, 256);
        im.chunk_first = (uint32_t)chunk_img.size();
        im.n_chunks = (im.raw_len + kScanChunkBytes - 1) / kScanChunkBytes;
        for (uint32_t k = 0; k < im.n_chunks; k++) chunk_img.push_back((uint32_t)i);
        im.mcu_count = (uint32_t)d.mcu_count;
        im.mcu_count_w = (uint32_t)d.mcu_count_w;
        im.has_dri = d.restart_interval > 0 ? 1u : 0u;
        im.restart_interval = im.has_dri ? (uint32_t)d.restart_interval : im.mcu_count;
        im.seg_first = seg_total;
        im.n_segs = (im.mcu_count + im.restart_interval - 1) / im.restart_interval;
        seg_total += im.n_segs;
        if (coef_only) { /* no entropy stage: no decode CTAs of either kind */ }
        else if (im.has_dri)
            for (uint32_t s = 0; s < im.n_segs; s += kHuffThreads) ctas.push_back({(uint32_t)i, s});
        else
        {
            // no restart markers: self-synchronising sub-sequence decode, one lane per kSubBytes of stream
            im.sub_first = sub_total;
            im.scta_first = (uint32_t)sctas.size();
            im.n_sub_max = (im.raw_len + kSubBytes - 1) / kSubBytes;
            if (im.n_sub_max == 0) im.n_sub_max = 1;
            sub_total += im.n_sub_max;
            for (uint32_t s = 0; s < im.n_sub_max; s += kSyncLanes) sctas.push_back({(uint32_t)i, s});   // one chunk per CTA
            simgs.push_back((uint32_t)i);
        }
        im.blk_first = (uint32_t)blk_total;
        im.blk_count = (uint32_t)d.blk_count;
        blk_total += (size_t)d.blk_count;
        im.width = (uint32_t)d.width;
        im.height = (uint32_t)d.height;
        im.mode = mode_of(d);
        im.tot_blks = (uint32_t)d.tot_blks_per_mcu;
        im.ny_blks = (uint32_t)d.blks_per_mcu[0];
        im.nu_blks = (uint32_t)d.blks_per_mcu[1];
        im.samp = (uint32_t)(d.sampling[0] >> 4) | (uint32_t)(d.sampling[0] & 0xF) << 4;
        // a gray frame has no chroma: geometry_ok() does not look at sampling[1..2] then, and the kernels that derive the
        // block layout from samp (the generic and the libjpeg-model ones) must see zero blocks there
        if (im.mode != kModeGray)
            im.samp |= (uint32_t)(d.sampling[1] >> 4) << 8 | (uint32_t)(d.sampling[1] & 0xF) << 12 | (uint32_t)(d.sampling[2] >> 4) << 16 |
                       (uint32_t)(d.sampling[2] & 0xF) << 20;
        im.yh = (uint32_t)(d.sampling[0] >> 4);
        const uint32_t mcus_per_tile = kTileBlocks / im.tot_blks;
        for (uint32_t m = 0; m < im.mcu_count; m += mcus_per_tile)
        {
            const uint32_t n = im.mcu_count - m < mcus_per_tile ? im.mcu_count - m : mcus_per_tile;
            tiles.push_back({(uint32_t)i, m, im.blk_first + m * im.tot_blks, im.mode | (n << 8)});
        }
        // quantisers: file (zig-zag) order -> natural order, per component (decoder.cpp:315,340)
        for (int c = 0; c < 3; c++)
            for (int k = 0; k < 64; k++)
            {
                const uint16_t q = coef_only ? (uint16_t)1 : d.quant[d.quant_id[c]][k];
                qtabs[(size_t)i * 192 + (size_t)c * 64 + zz[k]] = q;
                if (q > 255) im.wide_q = 1;
            }
        pixels += (int64_t)d.width * d.height;
        if (coef_only) continue;
        scan_bytes += (int64_t)d.scan_size;
        // decode tables, shared between images that carry identical DHT payloads
        std::string key;
        for (int c = 0; c < 3; c++)
        {
            const int slots[2] = {d.huff_id[c] >> 4, 4 + (d.huff_id[c] & 0xF)};
            for (int s = 0; s < 2; s++)
            {
                if (slots[s] < 0 || slots[s] > 7 || !d.huff_present[slots[s]]) { rc = B2J_E_UNSUPPORTED; break; }
                key.append((const char *)d.huff_counts[slots[s]], 16);
                size_t tot = 0;
                for (int l = 0; l < 16; l++) tot += d.huff_counts[slots[s]][l];
                key.append((const char *)d.huff_symbols[slots[s]], tot);
                key.push_back((char)0xA5);
            }
        }
        if (rc != B2J_OK) break;
        auto it = lut_cache.find(key);
        if (it == lut_cache.end())
        {
            std::vector<uint16_t> set;
            if (!build_lut_set(d, set)) { rc = B2J_E_UNSUPPORTED; t_last_error = "Huffman tables need more decode-table space than one CTA has"; break; }
            const uint32_t off = (uint32_t)luts.size();
            luts.insert(luts.end(), set.begin(), set.end());
            it = lut_cache.emplace(key, LutRef{off, (uint32_t)set.size(), (uint32_t)set[12]}).first;
        }
        im.lut_off = it->second.off;
        im.lut_len = it->second.len;
        im.lut_dec_len = it->second.dec_len;
        if (im.lut_len > max_lut_len) max_lut_len = im.lut_len;
        if (im.lut_dec_len > max_lut_dec_len) max_lut_dec_len = im.lut_dec_len;
        if (im.lut_len - im.lut_dec_len > max_lut_walk_len) max_lut_walk_len = im.lut_len - im.lut_dec_len;
    }
    if (rc != B2J_OK) { delete b; return rc; }
    if (blk_total + kTileBlocks >= 0xFFFFFFF0ull) { delete b; return B2J_E_ARG; }
    // tiles sorted by kind, each kind a kernel of its own: the four everyday colour layouts, one-component images, the rest
    const auto gray0 = std::stable_partition(tiles.begin(), tiles.end(), [](const TileDev &t) { return (t.info & 0xFFu) < kModeGray; });
    const auto generic0 = std::stable_partition(gray0, tiles.end(), [](const TileDev &t) { return (t.info & 0xFFu) == kModeGray; });

    // ---- input blob layout: regions 256-byte aligned, in this order; a region of no bytes shares its offset with the next
    size_t off = 0;
    auto place = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
    auto place_array = [&](const auto &v) { return place(sizeof(v[0]) * v.size()); };
    const size_t o_imgs = place_array(b->imgs);
    const size_t o_chunk_img = place_array(chunk_img);
    const size_t o_ctas = place_array(ctas);
    const size_t o_sctas = place_array(sctas);
    const size_t o_simgs = place_array(simgs);
    const size_t o_tiles = place_array(tiles);
    const size_t o_luts = place_array(luts);
    const size_t o_qtabs = place_array(qtabs);
    const size_t o_raw = place(raw_total + kScanChunkBytes + 64);   // the pre-pass reads whole chunks
    b->blob_bytes = off;

    // ---- scratch layout
    off = 0;
    const size_t o_clean = place(raw_total + 256);   // the bit readers prefetch up to 48 bytes past a segment
    b->clean_bytes = off - o_clean;
    const size_t o_clean_len = place(4 * (size_t)n);
    const size_t o_seg_start = place(4 * (size_t)seg_total);
    const size_t o_recs = place(sizeof(SubRec) * (size_t)sub_total);
    const size_t o_pres = place(sizeof(uint4) * (sctas.size() + 1));
    const size_t o_chunk_states = place(sizeof(uint4) * (sctas.size() + 1));
    // what every decode starts from zero, side by side: one memset
    const size_t o_status = place(4 * (size_t)n);
    const size_t o_scan_cut = place(4 * (size_t)n);
    const size_t o_sync_stats = place(4 * 8);
    const size_t o_chunk_state = place(8 * chunk_img.size());
    b->zero_bytes = off - o_status;
    const size_t scratch_bytes = off;
    b->n_segs_total = seg_total;
    b->coef_rows = blk_total + kTileBlocks;   // one tile of padding: the last tile may read past the last block

    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        cudaError_t e;
        if ((e = ctx->pin_pool.get(b->blob_bytes, b->h_blob)) != cudaSuccess ||
            (e = ctx->dev_pool.get(b->blob_bytes, b->d_blob)) != cudaSuccess ||
            (e = ctx->dev_pool.get(scratch_bytes, b->d_scratch)) != cudaSuccess ||
            (e = ctx->dev_pool.get(b->coef_rows * 128, b->d_coef)) != cudaSuccess ||
            (e = ctx->dev_pool.get(pix_total, b->d_pix)) != cudaSuccess)
        {
            rc = fail_cuda(e, "batch allocation");
            cudaGetLastError();
        }
    }
    if (rc != B2J_OK) { release_batch_buffers(b); delete b; return rc == B2J_E_CUDA ? B2J_E_NOMEM : rc; }
    rc = make_tensor_map(ctx, b);
    if (rc != B2J_OK) { release_batch_buffers(b); delete b; return rc; }

    // ---- the pinned blob, and where the kernels find each region on the device
    DecodeArgs &a = b->args;
    a.imgs = stage(b, o_imgs, b->imgs);
    b->h_imgs = at<ImgDev>(b->h_blob, o_imgs);
    a.chunk_img = stage(b, o_chunk_img, chunk_img);
    a.huff_ctas = stage(b, o_ctas, ctas);
    a.sync_ctas = stage(b, o_sctas, sctas);
    a.sync_imgs = stage(b, o_simgs, simgs);
    a.tiles = stage(b, o_tiles, tiles);
    a.luts = stage(b, o_luts, luts);
    a.qtabs = stage(b, o_qtabs, qtabs);
    for (int i = 0; i < n; i++)
    {
        const ImgDev &im = b->imgs[(size_t)i];
        uint8_t *dst = at<uint8_t>(b->h_blob, o_raw + im.raw_off);
        if (im.raw_len) memcpy(dst, files[i] + descs[i].scan_offset, im.raw_len);
        // pad with FF D9 D9 ...: running off the end of a scan then looks like EOI to the pre-pass
        memset(dst + im.raw_len, 0xD9, align_up((size_t)im.raw_len + 32, 16) - im.raw_len);
        dst[im.raw_len] = 0xFF;
    }
    a.raw = at<const uint8_t>(b->d_blob, o_raw);
    a.clean = at<uint8_t>(b->d_scratch, o_clean);
    a.clean_len = at<uint32_t>(b->d_scratch, o_clean_len);
    a.seg_start = at<uint32_t>(b->d_scratch, o_seg_start);
    a.recs = at<SubRec>(b->d_scratch, o_recs);
    a.sync_cta_base = at<uint4>(b->d_scratch, o_pres);
    a.sync_chunk_state = at<uint4>(b->d_scratch, o_chunk_states);
    a.status = at<int32_t>(b->d_scratch, o_status);
    a.scan_cut = at<uint32_t>(b->d_scratch, o_scan_cut);
    a.sync_stats = at<uint32_t>(b->d_scratch, o_sync_stats);
    a.chunk_state = at<uint64_t>(b->d_scratch, o_chunk_state);
    a.tmap = &b->tmap;
    a.coef = at<int16_t>(b->d_coef, 0);
    a.pixels = at<uint8_t>(b->d_pix, 0);
    a.n_images = (uint32_t)n;
    a.n_chunks = (uint32_t)chunk_img.size();
    a.n_huff_ctas = (uint32_t)ctas.size();
    a.n_sync_ctas = (uint32_t)sctas.size();
    a.n_sync_imgs = (uint32_t)simgs.size();
    a.gray_tile0 = (uint32_t)(gray0 - tiles.begin());
    a.generic_tile0 = (uint32_t)(generic0 - tiles.begin());
    a.n_tiles = (uint32_t)tiles.size();
    a.max_lut_len = max_lut_len;
    a.max_lut_dec_len = max_lut_dec_len;
    a.max_lut_walk_len = max_lut_walk_len;
    a.any_wide_q = false;
    for (const ImgDev &im : b->imgs) a.any_wide_q = a.any_wide_q || im.wide_q != 0;
    a.samples = nullptr;
    {
        const char *sp = getenv("B2J_SYNC_PRE");
        a.sync_use_pre = !(sp && atoi(sp) == 0);
    }

    b2j_batch_info &inf = b->info;
    memset(&inf, 0, sizeof(inf));
    inf.n_images = n;
    inf.total_pixels = pixels;
    inf.total_blocks = (int64_t)blk_total;
    inf.scan_bytes = scan_bytes;
    inf.coef_plane_bytes = 128 * (int64_t)blk_total;
    inf.pixel_bytes = 4 * pixels;
    inf.algorithmic_bytes = inf.scan_bytes + 2 * inf.coef_plane_bytes + inf.pixel_bytes;
    inf.device_bytes = device_bytes(b);
    inf.h2d_bytes = (int64_t)b->blob_bytes;
    b->fixed_launches = 1 + (ctas.empty() ? 0 : 1) + (sctas.empty() ? 0 : kSyncLaunches);
    set_output(b, B2J_PIXELS_REFERENCE, B2J_OUT_BGRA, 1);
    *out = b;
    return B2J_OK;
}

extern "C" void b2j_batch_destroy(b2j_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    // the buffers go back to the pool: nothing enqueued on them may still be in flight, including work on a caller's stream
    if (b->last_stream && b->last_stream != b->ctx->stream) cudaStreamSynchronize(b->last_stream);
    cudaStreamSynchronize(b->ctx->stream);
    release_batch_buffers(b);
    delete b;
}

extern "C" int b2j_batch_get_info(const b2j_batch *b, b2j_batch_info *info)
{
    if (!b || !info) return B2J_E_ARG;
    *info = b->info;
    return B2J_OK;
}

extern "C" int b2j_batch_upload(b2j_batch *b, void *stream)
{
    if (!b) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, stream);
    CU_TRY(cudaMemcpyAsync(b->d_blob.p, b->h_blob.p, b->blob_bytes, cudaMemcpyHostToDevice, s));
    if (!b->uploaded)
    {
        // padding rows of the plane and the tail of the clean stream are read (never used); define them once
        CU_TRY(cudaMemsetAsync(b->args.coef + (b->coef_rows - kTileBlocks) * 64, 0, (size_t)kTileBlocks * 128, s));
        CU_TRY(cudaMemsetAsync(b->args.clean, 0, b->clean_bytes, s));
        b->uploaded = true;
    }
    return B2J_OK;
}

// Events of one timed step: start (before the memsets), before the pre-pass, after it, after the entropy stage,
// after the IDCT/colour stage (= end of the step).
constexpr size_t kStepEvents = 5;

// The orientation pass's tile table for the current settings, copied to the front of d_orient on `s`: one tile of
// kOrientTile x kOrientTile pixels per piece of every image whose code is not 1 (of its window when it is cropped), at
// the batch's scale.
static int stage_orient_tiles(b2j_batch *b, cudaStream_t s)
{
    // the pinned table is rebuilt only once the copy out of it has left
    if (!b->orient_copied) CU_TRY(cudaEventCreateWithFlags(&b->orient_copied, cudaEventDisableTiming));
    else CU_TRY(cudaEventSynchronize(b->orient_copied));
    OrientTileDev *t = at<OrientTileDev>(b->h_orient, 0);
    uint32_t k = 0;
    for (size_t i = 0; i < b->orient.size(); i++)
    {
        const uint32_t code = b->orient[i];
        if (code == 1) continue;
        const CropDev o = image_out(b, i).win;
        for (uint32_t ty = 0; ty * kOrientTile < o.h; ty++)
            for (uint32_t tx = 0; tx * kOrientTile < o.w; tx++) t[k++] = {b->orient_off[i], (uint32_t)i, tx | ty << 11 | code << 22};
    }
    b->n_orient_tiles = k;
    CU_TRY(cudaMemcpyAsync(b->d_orient.p, t, sizeof(OrientTileDev) * k, cudaMemcpyHostToDevice, s));
    CU_TRY(cudaEventRecord(b->orient_copied, s));
    b->orient_stale = false;
    return B2J_OK;
}

// The crop windows, the window views and the crop tile list for the current settings, copied to d_crop on `s`. GRAY8
// and scale 1/8 have no fancy upsampling, so their tiles need no halo. A tile's TMA box is always kTileBlocks rows from
// its first block, which lies inside the plane: it ends inside the plane's kTileBlocks rows of slack (coef_rows).
static int stage_crop_tiles(b2j_batch *b, cudaStream_t s)
{
    // the pinned copy is rebuilt only once the copy out of it has left
    if (!b->crop_copied) CU_TRY(cudaEventCreateWithFlags(&b->crop_copied, cudaEventDisableTiming));
    else CU_TRY(cudaEventSynchronize(b->crop_copied));
    const uint32_t halo = (b->args.out_format == B2J_OUT_GRAY8 || b->args.scale == 8) ? 0u : 1u;
    CropDev *w = at<CropDev>(b->h_crop, 0);
    ImgDev *v = at<ImgDev>(b->h_crop, b->crop_views_off);
    std::vector<TileDev> tiles;
    for (size_t i = 0; i < b->imgs.size(); i++)
    {
        w[i] = b->win[i];
        v[i] = b->imgs[i];
        v[i].width = w[i].w;
        v[i].height = w[i].h;
        crop_tiles(b->imgs[i], (uint32_t)i, w[i], b->args.scale, halo, tiles);
    }
    memcpy(at<TileDev>(b->h_crop, b->crop_tiles_off), tiles.data(), sizeof(TileDev) * tiles.size());
    b->args.n_crop_tiles = (uint32_t)tiles.size();
    CU_TRY(cudaMemcpyAsync(b->d_crop.p, b->h_crop.p, b->crop_tiles_off + sizeof(TileDev) * tiles.size(), cudaMemcpyHostToDevice, s));
    CU_TRY(cudaEventRecord(b->crop_copied, s));
    b->crop_stale = false;
    return B2J_OK;
}

// One decode of the whole batch: the pre-pass, the entropy stage and the IDCT/colour stage, in order on `s`, then the
// orientation pass when some image's code is not 1.
static int enqueue_decode(b2j_batch *b, cudaStream_t s, cudaEvent_t *ev /* kStepEvents or NULL */)
{
    if (!b->uploaded) { t_last_error = "b2j_batch_decode before b2j_batch_upload"; return B2J_E_ARG; }
    if (const char *why = output_refusal(b->args.pixel_model, b->args.out_format, (int)b->args.scale, !b->crops.empty())) { t_last_error = why; return B2J_E_ARG; }
    if (const int rc = crop_refusal(b)) return rc;
    if (b->args.pixel_model == B2J_PIXELS_LIBJPEG && b->args.out_format != B2J_OUT_GRAY8 && !b->d_samples.p)
    {
        // the sample plane: 64 bytes per block, image by image at 64 * blk_first
        const cudaError_t e = grow(b->ctx, b->d_samples, (size_t)b->info.total_blocks * 64);
        if (e != cudaSuccess) { fail_cuda(e, "sample plane allocation"); return B2J_E_NOMEM; }
        b->args.samples = at<uint8_t>(b->d_samples, 0);
        b->info.device_bytes = device_bytes(b);
    }
    if (b->orient_stale)
        if (const int rc = stage_orient_tiles(b, s)) return rc;
    if (b->crop_stale)
        if (const int rc = stage_crop_tiles(b, s)) return rc;
    const DecodeArgs &a = b->args;
    if (ev) CU_TRY(cudaEventRecord(ev[0], s));
    if (a.n_huff_ctas) CU_TRY(cudaMemsetAsync(a.seg_start, 0xFF, 4 * (size_t)b->n_segs_total, s));   // read by the restart-interval decoder only
    CU_TRY(cudaMemsetAsync(a.status, 0, b->zero_bytes, s));   // status words, sync stats, look-back words
    if (ev) CU_TRY(cudaEventRecord(ev[1], s));
    launch_prepass(a, s);
    if (ev) CU_TRY(cudaEventRecord(ev[2], s));
    launch_huffman(a, s);
    launch_huffman_sync(a, s);
    if (ev) CU_TRY(cudaEventRecord(ev[3], s));
    launch_idct(a, s);
    // a cropped image is oriented as an image of its window's size: the window views at scale 1
    if (!b->orient.empty())
        launch_orient(a.pixels, a.crops ? at<const ImgDev>(b->d_crop, b->crop_views_off) : a.imgs, at<const OrientTileDev>(b->d_orient, 0), b->n_orient_tiles,
                      a.crops ? 1u : a.scale, a.out_format, at<uint8_t>(b->d_orient, 0), s);
    if (ev) CU_TRY(cudaEventRecord(ev[4], s));
    CU_TRY(cudaGetLastError());
    return B2J_OK;
}

static void collect_times(cudaEvent_t *ev, b2j_stage_times *t)
{
    t->prepass_ms = t->huffman_ms = t->idct_ms = 0.f;
    cudaEventElapsedTime(&t->prepass_ms, ev[1], ev[2]);
    cudaEventElapsedTime(&t->huffman_ms, ev[2], ev[3]);
    cudaEventElapsedTime(&t->idct_ms, ev[3], ev[4]);
    cudaEventElapsedTime(&t->total_ms, ev[0], ev[4]);
}

extern "C" int b2j_batch_decode(b2j_batch *b, void *stream)
{
    if (!b) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    return enqueue_decode(b, pick_stream(b, stream), nullptr);
}

extern "C" int b2j_batch_decode_timed(b2j_batch *b, void *stream, b2j_stage_times *times)
{
    return b2j_batch_decode_steps(b, stream, 1, times, nullptr);
}

extern "C" int b2j_batch_decode_steps(b2j_batch *b, void *stream, int steps, b2j_stage_times *per_step, float *total_ms)
{
    if (!b || steps <= 0) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, stream);
    const size_t per = kStepEvents;
    std::vector<cudaEvent_t> ev((size_t)steps * per, nullptr);
    int rc = B2J_OK;
    for (auto &e : ev)
    {
        const cudaError_t ce = cudaEventCreate(&e);
        if (ce != cudaSuccess) { rc = fail_cuda(ce, "cudaEventCreate"); e = nullptr; break; }
    }
    for (int k = 0; k < steps && rc == B2J_OK; k++) rc = enqueue_decode(b, s, &ev[(size_t)k * per]);
    if (rc == B2J_OK)
    {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) rc = fail_cuda(e, "cudaStreamSynchronize");
    }
    if (rc == B2J_OK)
    {
        for (int k = 0; k < steps && per_step; k++) collect_times(&ev[(size_t)k * per], &per_step[k]);
        if (total_ms) cudaEventElapsedTime(total_ms, ev[0], ev[(size_t)steps * per - 1]);
    }
    for (auto &e : ev) if (e) cudaEventDestroy(e);
    return rc;
}

extern "C" int b2j_batch_sync(b2j_batch *b, void *stream)
{
    if (!b) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    CU_TRY(cudaStreamSynchronize(pick_stream(b, stream)));
    return B2J_OK;
}

extern "C" int b2j_batch_status(b2j_batch *b, void *stream, int32_t *status)
{
    if (!b || !status) return B2J_E_ARG;
    return read_back(b, stream, status, b->args.status, 4 * (size_t)b->n);
}

extern "C" int b2j_batch_sync_stats(b2j_batch *b, void *stream, uint32_t *out8)
{
    if (!b || !out8) return B2J_E_ARG;
    return read_back(b, stream, out8, b->args.sync_stats, 4 * 8);
}

extern "C" int b2j_batch_set_output_format(b2j_batch *b, int format)
{
    if (!b || !format_ok(format)) return B2J_E_ARG;
    set_output(b, b->args.pixel_model, format, (int)b->args.scale);
    return B2J_OK;
}

extern "C" int b2j_batch_set_pixel_model(b2j_batch *b, int model)
{
    if (!b || !model_ok(model)) return B2J_E_ARG;
    set_output(b, model, b->args.out_format, (int)b->args.scale);
    return B2J_OK;
}

extern "C" int b2j_batch_set_scale(b2j_batch *b, int denom)
{
    if (!b || !scale_ok(denom)) return B2J_E_ARG;
    set_output(b, b->args.pixel_model, b->args.out_format, denom);
    return B2J_OK;
}

extern "C" int b2j_batch_set_orientations(b2j_batch *b, const uint8_t *codes)
{
    if (!b) return B2J_E_ARG;
    bool any = false;
    for (int i = 0; codes && i < b->n; i++)
    {
        if (codes[i] < 1 || codes[i] > 8) return B2J_E_ARG;
        any = any || codes[i] != 1;
    }
    CU_TRY(cudaSetDevice(b->ctx->device));
    // the buffers go back to the pool or grow: work in flight may still read the table or write the copies
    if (b->last_stream && (b->d_orient.p || any)) CU_TRY(cudaStreamSynchronize(b->last_stream));
    b->orient.clear();
    b->orient_off.clear();
    b->orient_table_bytes = 0;
    int rc = B2J_OK;
    if (any)
    {
        size_t tiles = 0, bytes = 0;   // at scale 1 in BGRA, the most any setting needs
        for (int i = 0; i < b->n; i++)
            if (codes[i] != 1)
            {
                const Dims o = out_dims(b->imgs[(size_t)i], 1);
                tiles += (size_t)((o.w + kOrientTile - 1) / kOrientTile) * ((o.h + kOrientTile - 1) / kOrientTile);
                bytes += (size_t)o.w * o.h * 4 + pack_align(B2J_OUT_BGRA) - 1;
            }
        const size_t table = align_up(sizeof(OrientTileDev) * tiles, 256);
        if (grow(b->ctx, b->d_orient, table + bytes) != cudaSuccess || grow(b->ctx, b->h_orient, table, true) != cudaSuccess)
        {
            t_last_error = "orientation buffer allocation";
            rc = B2J_E_NOMEM;   // every code is 1 then
        }
        else
        {
            b->orient.assign(codes, codes + b->n);
            b->orient_off.assign((size_t)b->n, 0);
            b->orient_table_bytes = table;
        }
    }
    if (b->orient.empty()) release_orient_buffers(b);
    b->info.device_bytes = device_bytes(b);
    set_output(b, b->args.pixel_model, b->args.out_format, (int)b->args.scale);
    return rc;
}

extern "C" int b2j_batch_set_crops(b2j_batch *b, const int32_t *boxes)
{
    if (!b) return B2J_E_ARG;
    for (int i = 0; boxes && i < b->n; i++)
        if (boxes[4 * i] < 0 || boxes[4 * i + 1] < 0 || boxes[4 * i + 2] < 1 || boxes[4 * i + 3] < 1) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    // the buffers go back to the pool or grow: work in flight may still read the windows or the tiles
    if (b->last_stream && (b->d_crop.p || boxes)) CU_TRY(cudaStreamSynchronize(b->last_stream));
    b->crops.clear();
    b->win.clear();
    int rc = B2J_OK;
    if (boxes)
    {
        size_t tiles = 0;   // at any window and scale
        for (const ImgDev &im : b->imgs) tiles += crop_tiles_max(im);
        b->crop_views_off = align_up(sizeof(CropDev) * (size_t)b->n, 256);
        b->crop_tiles_off = b->crop_views_off + align_up(sizeof(ImgDev) * (size_t)b->n, 256);
        const size_t bytes = b->crop_tiles_off + sizeof(TileDev) * tiles;
        if (grow(b->ctx, b->d_crop, bytes) != cudaSuccess || grow(b->ctx, b->h_crop, bytes, true) != cudaSuccess)
        {
            t_last_error = "crop buffer allocation";
            rc = B2J_E_NOMEM;   // no crops then
        }
        else
        {
            b->crops.assign(boxes, boxes + 4 * (size_t)b->n);
            b->win.assign((size_t)b->n, CropDev{});
        }
    }
    if (b->crops.empty()) release_crop_buffers(b);
    b->info.device_bytes = device_bytes(b);
    set_output(b, b->args.pixel_model, b->args.out_format, (int)b->args.scale);
    return rc;
}

extern "C" int b2j_batch_pixels_device(const b2j_batch *b, int image, void **dptr, size_t *nbytes)
{
    if (!image_of(b, image) || !dptr) return B2J_E_ARG;
    if (const int rc = crop_refusal(b)) return rc;
    *dptr = result_of(b, (size_t)image);
    if (nbytes) *nbytes = image_bytes(b, (size_t)image);
    return B2J_OK;
}

extern "C" int b2j_batch_coefs_device(const b2j_batch *b, int image, void **dptr, size_t *nbytes)
{
    const ImgDev *im = image_of(b, image);
    if (!im || !dptr) return B2J_E_ARG;
    *dptr = b->args.coef + (size_t)im->blk_first * 64;
    if (nbytes) *nbytes = (size_t)im->blk_count * 128;
    return B2J_OK;
}

extern "C" int b2j_batch_read_pixels(b2j_batch *b, void *stream, int image, uint8_t *dst)
{
    if (!image_of(b, image) || !dst) return B2J_E_ARG;
    if (const int rc = crop_refusal(b)) return rc;
    return read_back(b, stream, dst, result_of(b, (size_t)image), image_bytes(b, (size_t)image));
}

extern "C" int b2j_batch_read_all_pixels(b2j_batch *b, void *stream, uint8_t *const *dsts)
{
    if (!b || !dsts) return B2J_E_ARG;
    if (const int rc = crop_refusal(b)) return rc;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, stream);
    for (int i = 0; i < b->n; i++)
    {
        if (!dsts[i]) continue;
        CU_TRY(cudaMemcpyAsync(dsts[i], result_of(b, (size_t)i), image_bytes(b, (size_t)i), cudaMemcpyDeviceToHost, s));
    }
    CU_TRY(cudaStreamSynchronize(s));
    return B2J_OK;
}

extern "C" int b2j_batch_read_coefs(b2j_batch *b, void *stream, int image, int32_t *dst)
{
    const ImgDev *im = image_of(b, image);
    if (!im || !dst) return B2J_E_ARG;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, stream);
    const size_t bytes = (size_t)im->blk_count * 256;
    const cudaError_t e = grow(b->ctx, b->d_expand, bytes);
    if (e != cudaSuccess) return fail_cuda(e, "coefficient tap allocation");
    launch_expand(b->args.coef + (size_t)im->blk_first * 64, b->args.qtabs + (size_t)image * 192, im->blk_count, im->tot_blks, im->ny_blks, im->nu_blks,
                  at<int32_t>(b->d_expand, 0), s);
    CU_TRY(cudaGetLastError());
    return read_back(b, stream, dst, b->d_expand.p, bytes);
}

// ---------------------------------------------------------------------------------------
// Output stage: reduced copies of the decoded pixels (SURVEY.md 8f rank 3).
extern "C" int b2j_batch_downscale(b2j_batch *b, void *stream, int factor)
{
    if (!b || (factor != 2 && factor != 4 && factor != 8)) return B2J_E_ARG;
    if (b->args.scale != 1) { t_last_error = "b2j_batch_downscale of a scaled decode"; return B2J_E_ARG; }
    // k_downscale takes each image's size from its unoriented descriptor
    if (!b->orient.empty()) { t_last_error = "b2j_batch_downscale of oriented images (b2j_batch_set_orientations)"; return B2J_E_ARG; }
    if (!b->crops.empty()) { t_last_error = "b2j_batch_downscale of cropped images (b2j_batch_set_crops)"; return B2J_E_ARG; }
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, stream);
    const int fmt = b->args.out_format;
    if (b->small_factor != factor)
    {
        b->small_factor = 0;   // no reduced copy until the buffer and its offset table are in place
        b->small_off.resize((size_t)b->n);
        size_t off = align_up(8 * (size_t)b->n, 256);   // behind the offset table
        for (int i = 0; i < b->n; i++)
        {
            const Dims o = out_dims(b->imgs[(size_t)i], (uint32_t)factor);
            b->small_off[(size_t)i] = off;
            off += align_up((size_t)o.w * o.h * format_bpp(B2J_OUT_BGRA), 16);   // sized for BGRA: every format fits
        }
        if (grow(b->ctx, b->d_small, off) != cudaSuccess) return B2J_E_NOMEM;
        CU_TRY(cudaMemcpyAsync(b->d_small.p, b->small_off.data(), 8 * (size_t)b->n, cudaMemcpyHostToDevice, s));
        CU_TRY(cudaStreamSynchronize(s));   // the table is a pageable vector that may be rebuilt
        b->small_factor = factor;
    }
    uint32_t max_samples = 0;
    for (const ImgDev &im : b->imgs)
    {
        const Dims o = out_dims(im, (uint32_t)factor);
        max_samples = std::max(max_samples, o.w * o.h * (fmt == B2J_OUT_RGB_PLANAR ? 3u : 1u));
    }
    launch_downscale(b->args.pixels, b->args.imgs, at<const uint64_t>(b->d_small, 0), at<uint8_t>(b->d_small, 0), (uint32_t)b->n, max_samples,
                     (uint32_t)factor, fmt, s);
    CU_TRY(cudaGetLastError());
    return B2J_OK;
}

extern "C" int b2j_batch_downscaled_device(const b2j_batch *b, int image, void **dptr, size_t *nbytes, int *width, int *height)
{
    const ImgDev *im = image_of(b, image);
    if (!im || !dptr || !b->small_factor) return B2J_E_ARG;
    const Dims o = out_dims(*im, (uint32_t)b->small_factor);
    *dptr = at<uint8_t>(b->d_small, b->small_off[(size_t)image]);
    if (nbytes) *nbytes = (size_t)o.w * o.h * format_bpp(b->args.out_format);
    if (width) *width = (int)o.w;
    if (height) *height = (int)o.h;
    return B2J_OK;
}

extern "C" int b2j_batch_read_downscaled(b2j_batch *b, void *stream, int image, uint8_t *dst)
{
    void *p = nullptr; size_t nb = 0;
    if (!dst) return B2J_E_ARG;
    const int rc = b2j_batch_downscaled_device(b, image, &p, &nb, nullptr, nullptr);
    return rc != B2J_OK ? rc : read_back(b, stream, dst, p, nb);
}

// ---------------------------------------------------------------------------------------
// Host feed (SURVEY.md 8f rank 2/3): b2j_decode_host_ex / _multi, pinned buffers, file reader.

namespace {

// Host feed only: the images of the batch packed as tightly in the pixel plane as the stores of the colour kernel allow
// (pack_align), so that the downloads of neighbouring images merge into one copy when the caller's buffers are
// neighbours too. After set_output(), before b2j_batch_upload().
void pack_pixel_plane(b2j_batch *b)
{
    const size_t a = pack_align(b->args.out_format);
    size_t off = 0;
    for (size_t i = 0; i < b->imgs.size(); i++)
    {
        b->imgs[i].pix_off = off = align_up(off, a);
        off += image_bytes(b, i);
    }
    memcpy(b->h_imgs, b->imgs.data(), sizeof(ImgDev) * (size_t)b->n);
}

int auto_threads(int asked, int cap)
{
    if (asked > 0) return asked < 64 ? asked : 64;
    const unsigned hw = std::thread::hardware_concurrency();
    int t = hw ? (int)hw : 4;
    return t < cap ? t : cap;
}

struct FeedGroup
{
    int first = 0, count = 0;            // file index range
    b2j_batch *b = nullptr;              // built by a worker; nullptr when no file of the group was accepted
    std::vector<int> idx;                // file index of every image of the batch
    int rc = B2J_OK;
    std::string err;
    bool ready = false;                  // set by the worker under the feed mutex
    bool parsed = false;                 // the header verdicts of its files are in status[]
    cudaEvent_t decoded = nullptr, done = nullptr;
};

} // namespace

extern "C" int b2j_decode_host_crop(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, const b2j_host_opts *opts,
                                    const int32_t *crops, uint8_t *const *out, int32_t *status)
{
    if (!ctx || n <= 0 || !files || !lens || !out || !status || !opts) return B2J_E_ARG;
    const int fmt = opts->out_format, model = opts->pixel_model, scale = opts->scale ? opts->scale : 1;
    const bool orient = opts->exif_orientation == 1;
    if (!format_ok(fmt) || !model_ok(model) || !scale_ok(scale) || (opts->exif_orientation & ~1)) return B2J_E_ARG;
    if (const char *why = output_refusal(model, fmt, scale, crops != nullptr)) { t_last_error = why; return B2J_E_ARG; }
    CU_TRY(cudaSetDevice(ctx->device));
    const int gate = opts->gate;
    const int group = opts->group > 0 ? opts->group : 32;
    const int n_threads = auto_threads(opts->n_threads, 8);

    // Groups of consecutive files. The first groups are small (2, 4, 8, ...): nothing travels device->host before the
    // first group is parsed, staged, uploaded and decoded, so that lead time is kept short.
    // A group is also bounded in bytes: one worker stages a group's scans into pinned memory, and a group of large files
    // would hold the pipeline up for as long as that copy takes (32 x 6.7 MB of 4K scans: 20 ms and more; measured on 64 x 4K: 54.9 / 45.1 / 41.1 / 40.9 ms for bounds of 1024 / 48 / 12 / 6 MiB).
    const size_t group_bytes = (size_t)(opts->group_mb > 0 ? opts->group_mb : 12) << 20;
    std::vector<FeedGroup> groups;
    for (int next = 0, ramp = 2; next < n; ramp *= 2)
    {
        FeedGroup g;
        g.first = next;
        const int want = std::min(n - next, std::min(ramp, group));
        size_t bytes = 0;
        while (g.count < want && (g.count == 0 || bytes + lens[next + g.count] <= group_bytes)) bytes += lens[next + g.count++];
        next += g.count;
        groups.push_back(std::move(g));
        if (ramp > group) ramp = group;
    }
    const int ng = (int)groups.size();

    // per-image status words come back through one pinned array, copied behind each group's pixels
    PoolBuf h_status_buf;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->pin_pool.get(4 * (size_t)n, h_status_buf) != cudaSuccess) { cudaGetLastError(); return B2J_E_NOMEM; }
    }
    int32_t *const h_status = at<int32_t>(h_status_buf, 0);

    std::mutex mu;
    std::condition_variable cv;
    std::atomic<int> next_group(0);
    int consumed = 0;                    // groups the enqueueing thread has taken (under mu)
    bool stop = false;
    const int window = n_threads + 2;    // groups built ahead of the enqueueing thread: bounds the pinned staging in flight

    auto worker = [&]() {
        cudaSetDevice(ctx->device);
        std::vector<b2j_image_desc> d;
        std::vector<const uint8_t *> f;
        std::vector<size_t> l;
        std::vector<uint8_t> codes;   // orientation codes of the accepted files
        std::vector<int32_t> boxes;   // their crop boxes
        for (;;)
        {
            const int g = next_group.fetch_add(1);
            if (g >= ng) return;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || g < consumed + window; });
                if (stop) { groups[(size_t)g].ready = true; cv.notify_all(); continue; }
            }
            FeedGroup &G = groups[(size_t)g];
            d.clear(); f.clear(); l.clear(); codes.clear(); boxes.clear();
            for (int i = G.first; i < G.first + G.count; i++)
            {
                b2j_image_desc desc;
                const int prc = b2j_parse_header(files[i], lens[i], gate, &desc);
                status[i] = prc;
                if (prc != B2J_OK) continue;
                int32_t code = 1;
                if (orient) b2j_parse_orientation(files[i], lens[i], &code);
                if (crops)
                {
                    // the box must lie inside the image's frame at the scale, oriented; else the image is skipped
                    CropDev win;
                    const uint32_t fw = ((uint32_t)desc.width + scale - 1) / scale, fh = ((uint32_t)desc.height + scale - 1) / scale;
                    if (!crop_window(fw, fh, (uint32_t)code, crops + 4 * (size_t)i, win)) { status[i] = B2J_E_ARG; continue; }
                    boxes.insert(boxes.end(), crops + 4 * (size_t)i, crops + 4 * (size_t)i + 4);
                }
                G.idx.push_back(i); d.push_back(desc); f.push_back(files[i]); l.push_back(lens[i]);
                codes.push_back((uint8_t)code);
            }
            G.parsed = true;
            if (!d.empty())
            {
                G.rc = b2j_batch_create(ctx, (int)d.size(), d.data(), f.data(), l.data(), &G.b);
                if (G.rc == B2J_OK)
                {
                    set_output(G.b, model, fmt, scale);
                    if (orient) G.rc = b2j_batch_set_orientations(G.b, codes.data());
                    if (crops && G.rc == B2J_OK) G.rc = b2j_batch_set_crops(G.b, boxes.data());
                    pack_pixel_plane(G.b);
                }
                if (G.rc != B2J_OK) G.err = t_last_error;
            }
            {
                std::lock_guard<std::mutex> lk(mu);
                G.ready = true;
            }
            cv.notify_all();
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) pool.emplace_back(worker);

    int rc = B2J_OK;
    int oldest = 0;   // first group whose buffers are still held
    // Hands a group's status words to the caller and its buffers back to the pools; a second call does nothing.
    auto close_group = [&](FeedGroup &G) {
        if (G.b)
        {
            for (size_t k = 0; k < G.idx.size(); k++) status[G.idx[k]] = h_status[G.idx[k]];
            release_batch_buffers(G.b);   // no stream synchronisation: the group's work is over (its `done` event)
            delete G.b;
            G.b = nullptr;
        }
        if (G.decoded) cudaEventDestroy(G.decoded);
        if (G.done) cudaEventDestroy(G.done);
        G.decoded = G.done = nullptr;
    };
    // Closes the groups before `end`, oldest first, so that their buffers serve the groups still to come: with `wait`
    // once each group's downloads have arrived, without it up to the first group whose downloads are still in flight.
    auto retire = [&](int end, bool wait) {
        for (; oldest < end; oldest++)
        {
            FeedGroup &O = groups[(size_t)oldest];
            const cudaError_t q = !O.done ? cudaSuccess : (wait ? cudaEventSynchronize(O.done) : cudaEventQuery(O.done));
            if (!wait && q != cudaSuccess) { if (q == cudaErrorNotReady) cudaGetLastError(); return; }
            close_group(O);
        }
    };
    const int max_in_flight = window + 4;   // groups enqueued and not yet back: bounds the buffers the pools ever hold, so that
                                            // after the first call no group waits for a cudaMalloc / cudaHostAlloc
    for (int g = 0; g < ng && rc == B2J_OK; g++)
    {
        FeedGroup &G = groups[(size_t)g];
        retire(g - max_in_flight + 1, true);
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return G.ready; });
            consumed = g + 1;
        }
        cv.notify_all();
        if (G.rc != B2J_OK) { rc = G.rc; t_last_error = G.err; break; }
        if (!G.b) continue;
        if ((rc = b2j_batch_upload(G.b, ctx->stream)) != B2J_OK) break;
        if ((rc = b2j_batch_decode(G.b, ctx->stream)) != B2J_OK) break;
        cudaError_t e = cudaEventCreateWithFlags(&G.decoded, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&G.done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventRecord(G.decoded, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream2, G.decoded, 0);
        // one download per run of images that are neighbours on the device (in the pixel plane, or as oriented copies)
        // and in the caller's memory (a copy costs a few microseconds whatever its size: 8192 small images one by one
        // spend a third of the time on that)
        for (size_t k = 0; k < G.idx.size() && e == cudaSuccess;)
        {
            uint8_t *dst = out[G.idx[k]];
            const uint8_t *src = result_of(G.b, k);
            size_t bytes = image_bytes(G.b, k), k1 = k + 1;
            if (!dst) { k = k1; continue; }
            while (k1 < G.idx.size() && out[G.idx[k1]] == dst + bytes && result_of(G.b, k1) == src + bytes)
                bytes += image_bytes(G.b, k1++);
            e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream2);
            k = k1;
        }
        // the status words of the group's images land at their file indices (consecutive only when no file was refused)
        for (size_t k = 0; k < G.idx.size() && e == cudaSuccess;)
        {
            size_t k1 = k + 1;
            while (k1 < G.idx.size() && G.idx[k1] == G.idx[k1 - 1] + 1) k1++;
            e = cudaMemcpyAsync(h_status + G.idx[k], G.b->args.status + k, 4 * (k1 - k), cudaMemcpyDeviceToHost, ctx->stream2);
            k = k1;
        }
        if (e == cudaSuccess) e = cudaEventRecord(G.done, ctx->stream2);
        if (e != cudaSuccess) { rc = fail_cuda(e, "b2j_decode_host_crop enqueue"); break; }
        retire(g, false);
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
        consumed = ng;
    }
    cv.notify_all();
    for (auto &t : pool) t.join();
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream2);
    cudaError_t e1 = cudaStreamSynchronize(ctx->stream);
    cudaGetLastError();
    if (rc == B2J_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) rc = fail_cuda(e1 != cudaSuccess ? e1 : e2, "cudaStreamSynchronize");
    for (FeedGroup &G : groups)
    {
        // after a failure the status words of the groups in flight are not trustworthy: the header verdicts stay
        if (rc != B2J_OK) G.idx.clear();
        close_group(G);
        if (!G.parsed)   // only after a failure: every file still gets its header verdict
            for (int i = G.first; i < G.first + G.count; i++) { b2j_image_desc desc; status[i] = b2j_parse_header(files[i], lens[i], gate, &desc); }
    }
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->pin_pool.put(h_status_buf);
    }
    return rc;
}

extern "C" int b2j_decode_host_ex(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, const b2j_host_opts *opts,
                                  uint8_t *const *out, int32_t *status)
{
    return b2j_decode_host_crop(ctx, n, files, lens, opts, nullptr, out, status);
}

extern "C" int b2j_decode_host_multi(b2j_ctx *const *ctxs, int n_ctx, int n, const uint8_t *const *files, const size_t *lens,
                                     const b2j_host_opts *opts, uint8_t *const *out, int32_t *status)
{
    if (!ctxs || n_ctx <= 0 || n <= 0 || !files || !lens || !opts || !out || !status) return B2J_E_ARG;
    for (int k = 0; k < n_ctx; k++) if (!ctxs[k]) return B2J_E_ARG;
    // contiguous ranges of about equal compressed size (the decode time of an image follows its bytes)
    size_t total = 0;
    for (int i = 0; i < n; i++) total += lens[i];
    std::vector<int> cut((size_t)n_ctx + 1, n);
    cut[0] = 0;
    {
        size_t acc = 0;
        int k = 1;
        for (int i = 0; i < n && k < n_ctx; i++)
        {
            acc += lens[i];
            while (k < n_ctx && acc * (size_t)n_ctx >= total * (size_t)k) cut[(size_t)k++] = i + 1;
        }
    }
    std::vector<int> rcs((size_t)n_ctx, B2J_OK);
    std::vector<std::string> errs((size_t)n_ctx);
    std::vector<std::thread> th;
    b2j_host_opts o = *opts;
    if (o.n_threads <= 0) o.n_threads = std::max(1, auto_threads(0, 64) / n_ctx < 8 ? auto_threads(0, 64) / n_ctx : 8);
    for (int k = 0; k < n_ctx; k++)
    {
        const int a = cut[(size_t)k], b = cut[(size_t)k + 1];
        if (b <= a) continue;
        th.emplace_back([&, k, a, b]() {
            rcs[(size_t)k] = b2j_decode_host_ex(ctxs[k], b - a, files + a, lens + a, &o, out + a, status + a);
            if (rcs[(size_t)k] != B2J_OK) errs[(size_t)k] = t_last_error;
        });
    }
    for (auto &t : th) t.join();
    for (int k = 0; k < n_ctx; k++)
        if (rcs[(size_t)k] != B2J_OK) { t_last_error = errs[(size_t)k]; return rcs[(size_t)k]; }
    return B2J_OK;
}

extern "C" int b2j_host_alloc(void **out, size_t bytes)
{
    if (!out) return B2J_E_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) { *out = nullptr; const int rc = fail_cuda(e, "cudaHostAlloc"); cudaGetLastError(); return rc == B2J_E_CUDA ? B2J_E_NOMEM : rc; }
    return B2J_OK;
}

extern "C" void b2j_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

extern "C" int b2j_read_files(int n, const char *const *paths, int n_threads, void **arena, const uint8_t **files, size_t *lens)
{
    if (n <= 0 || !paths || !arena || !files || !lens) return B2J_E_ARG;
    *arena = nullptr;
    std::vector<size_t> off((size_t)n + 1, 0);
    int bad = 0;
    for (int i = 0; i < n; i++)
    {
        struct stat st;
        lens[i] = 0; files[i] = nullptr;
        if (paths[i] && stat(paths[i], &st) == 0 && S_ISREG(st.st_mode)) lens[i] = (size_t)st.st_size; else bad++;
        off[(size_t)i + 1] = off[(size_t)i] + align_up(lens[i], 64);
    }
    void *base = nullptr;
    const int rc = b2j_host_alloc(&base, off[(size_t)n] + 64);
    if (rc != B2J_OK) return rc;
    std::atomic<int> next(0), failed(0);
    auto reader = [&]() {
        for (;;)
        {
            const int i = next.fetch_add(1);
            if (i >= n) return;
            if (!lens[i]) continue;
            uint8_t *dst = (uint8_t *)base + off[(size_t)i];
            const int fd = open(paths[i], O_RDONLY);
            size_t got = 0;
            if (fd >= 0)
            {
                while (got < lens[i])
                {
                    const ssize_t r = pread(fd, dst + got, lens[i] - got, (off_t)got);
                    if (r <= 0) break;
                    got += (size_t)r;
                }
                close(fd);
            }
            if (got == lens[i]) files[i] = dst; else { lens[i] = 0; failed++; }
        }
    };
    const int nt = std::min(auto_threads(n_threads, 16), n);
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back(reader);
    for (auto &t : th) t.join();
    *arena = base;
    return (bad || failed.load()) ? B2J_E_ARG : B2J_OK;
}

// The reference's pixels with the default host feed.
extern "C" int b2j_decode_host(b2j_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, int gate,
                               uint8_t *const *out_bgra, int32_t *status)
{
    b2j_host_opts o;
    memset(&o, 0, sizeof(o));
    o.gate = gate;
    o.out_format = B2J_OUT_BGRA;
    return b2j_decode_host_ex(ctx, n, files, lens, &o, out_bgra, status);
}

// ---------------------------------------------------------------------------------------
// The secondary boundary (reference idct.h:9-18, oclDCT8x8.cpp): coefficients in, pixels out.

struct b2j_idct
{
    b2j_batch *b = nullptr;   // a coefficient-only batch of one image: tiles, unit quantisers, plane, pixels
    PoolBuf d_in;             // the uploaded int32 coefficients (kept: clidct_retrieve_data_from_device reads them back)
    int blk_count = 0;
};

extern "C" int b2j_idct_create(b2j_ctx *ctx, int width, int height, int luma_h, int luma_v, b2j_idct **out)
{
    if (!ctx || !out || width <= 0 || height <= 0 || luma_h < 1 || luma_h > 4 || luma_v < 1 || luma_v > 4) return B2J_E_ARG;
    *out = nullptr;
    b2j_image_desc d;
    memset(&d, 0, sizeof(d));
    d.width = width; d.height = height;
    d.sampling[0] = (uint8_t)((luma_h << 4) | luma_v); d.sampling[1] = d.sampling[2] = 0x11;
    d.color_space = (luma_h == 1 && luma_v == 1) ? B2J_CS_YUV444 : ((luma_h == 2 && luma_v == 2) ? B2J_CS_YUV411 : B2J_CS_OTHER);
    d.mcu_width = 8 * luma_h; d.mcu_height = 8 * luma_v;
    d.mcu_count_w = (width - 1) / d.mcu_width + 1; d.mcu_count_h = (height - 1) / d.mcu_height + 1;
    d.mcu_count = d.mcu_count_w * d.mcu_count_h;
    d.blks_per_mcu[0] = luma_h * luma_v; d.blks_per_mcu[1] = d.blks_per_mcu[2] = 1;
    d.tot_blks_per_mcu = luma_h * luma_v + 2;
    d.blk_count = d.mcu_count * d.tot_blks_per_mcu;
    b2j_idct *p = new b2j_idct;
    p->blk_count = d.blk_count;
    int rc = batch_create_impl(ctx, 1, &d, nullptr, nullptr, true, &p->b);
    if (rc == B2J_OK && grow(ctx, p->d_in, (size_t)d.blk_count * 256) != cudaSuccess) rc = B2J_E_NOMEM;
    if (rc == B2J_OK) rc = b2j_batch_upload(p->b, nullptr);   // descriptors, tiles, quantisers
    if (rc != B2J_OK) { b2j_idct_destroy(p); return rc; }
    *out = p;
    return B2J_OK;
}

extern "C" int b2j_idct_blk_count(const b2j_idct *p) { return p ? p->blk_count : B2J_E_ARG; }

extern "C" int b2j_idct_upload(b2j_idct *p, const int32_t *coefs, int offset, int count)
{
    if (!p || !coefs || offset < 0 || count < 0 || offset > p->blk_count || count > p->blk_count - offset) return B2J_E_ARG;
    b2j_batch *b = p->b;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, nullptr);
    int32_t *in = at<int32_t>(p->d_in, (size_t)offset * 256);
    CU_TRY(cudaMemcpyAsync(in, coefs, (size_t)count * 256, cudaMemcpyHostToDevice, s));
    launch_pack(in, b->args.coef + (size_t)offset * 64, (size_t)count * 64, s);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(s));   // the caller's buffer may be pageable and reused
    return B2J_OK;
}

extern "C" int b2j_idct_run(b2j_idct *p)
{
    if (!p) return B2J_E_ARG;
    b2j_batch *b = p->b;
    CU_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t s = pick_stream(b, nullptr);
    CU_TRY(cudaMemsetAsync(b->args.status, 0, 4, s));
    launch_idct(b->args, s);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(s));
    return B2J_OK;
}

extern "C" int b2j_idct_read_pixels(b2j_idct *p, uint8_t *dst)
{
    if (!p) return B2J_E_ARG;
    return b2j_batch_read_pixels(p->b, nullptr, 0, dst);
}

extern "C" int b2j_idct_read_coefs(b2j_idct *p, int32_t *dst)
{
    if (!p || !dst) return B2J_E_ARG;
    return read_back(p->b, nullptr, dst, p->d_in.p, (size_t)p->blk_count * 256);
}

extern "C" void b2j_idct_destroy(b2j_idct *p)
{
    if (!p) return;
    if (p->b)
    {
        b2j_ctx *ctx = p->b->ctx;
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        {
            std::lock_guard<std::mutex> lk(ctx->mu);
            ctx->dev_pool.put(p->d_in);
        }
        b2j_batch_destroy(p->b);
    }
    delete p;
}
