// kernels.h -- host-callable launchers of kernels.cu.
#ifndef B2J_KERNELS_H_INCLUDED
#define B2J_KERNELS_H_INCLUDED

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "b2j_internal.h"

namespace b2j {

struct DecodeArgs
{
    // inputs
    const uint8_t *raw;
    const ImgDev *imgs;
    const uint32_t *chunk_img;
    const HuffCtaDev *huff_ctas;   // restart-interval path: CTA -> (image, first segment)
    const HuffCtaDev *sync_ctas;   // self-synchronising path: CTA -> (image, first sub-sequence)
    const uint32_t *sync_imgs;     // images on the self-synchronising path
    const TileDev *tiles;
    const uint16_t *luts;
    const uint16_t *qtabs;
    const CUtensorMap *tmap;   // host copy, passed by value to the kernel
    // scratch
    uint8_t *clean;
    uint64_t *chunk_state;   // pre-pass: look-back words, zeroed before every decode
    uint32_t *clean_len, *seg_start;
    uint32_t *scan_cut;      // pre-pass: per image, ~(clean position of the first restart marker that starts no interval), zeroed before every decode
    SubRec *recs;           // self-synchronising path: one record per sub-sequence
    uint4 *sync_cta_base;   // per chunk (= decode CTA) of the self-synchronising path: (blocks started, DC sums), then their prefix
    uint4 *sync_chunk_state;   // per chunk: entry state it assumed (x, y), exit state (z, w)
    uint32_t *sync_stats;   // [r] = lanes that walked again in round r without meeting their checkpoint (r >= 6 in [6]), [7] = chunks the sweep re-ran
    bool sync_use_pre;      // pre-lanes on (default); off (B2J_SYNC_PRE=0): every chunk border is repaired by the sweep (test knob)
    // outputs
    int16_t *coef;
    uint8_t *pixels;
    int32_t *status;
    // sizes
    uint32_t n_images, n_chunks, n_huff_ctas, n_sync_ctas, n_sync_imgs, max_lut_len, max_lut_dec_len, max_lut_walk_len;   // LUT set lengths: whole / decode part / walk part
    // tiles, sorted by kind: [0, gray_tile0) the four everyday colour layouts, [gray_tile0, generic_tile0) one-component
    // images, [generic_tile0, n_tiles) every other layout (kModeGeneric)
    uint32_t gray_tile0, generic_tile0, n_tiles;
    int out_format;          // B2J_OUT_*: layout of the pixel plane (b2j_batch_set_output_format)
    bool any_wide_q;         // some quantiser of the batch exceeds 255 (16-bit DQT): generic dequantisation
    int pixel_model;         // B2J_PIXELS_*: which pixels the IDCT/colour stage computes (b2j_batch_set_pixel_model)
    uint8_t *samples;        // B2J_PIXELS_LIBJPEG: the sample plane, 64 B per block (allocated by the first decode in that model
                             // whose format is not B2J_OUT_GRAY8)
    uint32_t max_px_groups;  // largest ceil(OW / 4) * OH of the batch's output sizes: the grid of the libjpeg model's upsampling kernel
    uint32_t scale;          // B2J_PIXELS_LIBJPEG: the output is ceil(W / scale) x ceil(H / scale); 1, 2, 4 or 8 (b2j_batch_set_scale)
    // B2J_PIXELS_LIBJPEG, b2j_batch_set_crops: every image's window, nullptr = the whole images; the IDCT then runs over
    // the crop tile list (the windows' MCUs and their halo) instead of `tiles`
    const CropDev *crops;
    const TileDev *crop_tiles;
    uint32_t n_crop_tiles;
};

cudaError_t init_constants();
cudaError_t configure_kernels(uint32_t max_lut_len);
size_t huff_smem_bytes(uint32_t max_lut_len);
void launch_prepass(const DecodeArgs &a, cudaStream_t s);   // 1 kernel
void launch_huffman(const DecodeArgs &a, cudaStream_t s);   // 1 kernel
void launch_huffman_sync(const DecodeArgs &a, cudaStream_t s);   // 4 kernels
constexpr int kSyncLaunches = 4;
void launch_idct(const DecodeArgs &a, cudaStream_t s);      // reference model: 1 kernel per tile kind present; libjpeg model: 2, 1 in GRAY8
int idct_launches(const DecodeArgs &a);                      // kernels launch_idct() enqueues
void launch_downscale(const uint8_t *pix, const ImgDev *imgs, const uint64_t *out_off, uint8_t *out, uint32_t n_images, uint32_t max_out_samples,
                      uint32_t factor, int fmt, cudaStream_t s);   // box-filter reduction of the pixel plane
void launch_orient(const uint8_t *pix, const ImgDev *imgs, const OrientTileDev *tiles, uint32_t n_tiles, uint32_t scale, int fmt, uint8_t *out,
                   cudaStream_t s);   // 1 kernel: EXIF orientation of the images the tiles cover, into `out`
void launch_pack(const int32_t *in, int16_t *coef, size_t n_values, cudaStream_t s);   // int32 dequantised coefficients -> the int16 plane
void launch_expand(const int16_t *coef, const uint16_t *qtab, uint32_t blk_count, uint32_t tot, uint32_t ny, uint32_t nu, int32_t *out, cudaStream_t s);

} // namespace b2j
#endif
