// tests/native/cropcheck.cpp -- TEST INFRASTRUCTURE. Exposes the host side of a cropped decode (crop_plan.h: the box
// mapping through an orientation code and the crop tile list) to the CPU test-suite. Nothing here is a decode path.
#include <stdint.h>
#include <string.h>
#include <vector>

#include "crop_plan.h"

extern "C" {

// crop_window(): 1 and win[4] = x0, y0, w, h when the box fits, else 0.
int chk_crop_window(uint32_t fw, uint32_t fh, uint32_t code, const int32_t box[4], uint32_t win[4])
{
    b2j::CropDev w;
    if (!b2j::crop_window(fw, fh, code, box, w)) return 0;
    win[0] = w.x0; win[1] = w.y0; win[2] = w.w; win[3] = w.h;
    return 1;
}

// crop_tiles() of one image of mcw x mch MCUs (luma yh x yv blocks, tot blocks per MCU) for the window win: at most
// `cap` tiles as (first MCU, MCUs, first coefficient row) into out; returns the tile count. crop_tiles_max() in *max.
int chk_crop_tiles(uint32_t mcw, uint32_t mch, uint32_t yh, uint32_t yv, uint32_t tot, uint32_t blk_first, const uint32_t win[4], uint32_t scale,
                   uint32_t halo, uint32_t *out, int cap, long *max)
{
    b2j::ImgDev im;
    memset(&im, 0, sizeof(im));
    im.mcu_count_w = mcw;
    im.mcu_count = mcw * mch;
    im.samp = yh | yv << 4;
    im.tot_blks = tot;
    im.blk_first = blk_first;
    std::vector<b2j::TileDev> t;
    const b2j::CropDev w{win[0], win[1], win[2], win[3]};
    const uint32_t n = b2j::crop_tiles(im, 7, w, scale, halo, t);
    for (uint32_t k = 0; k < n && (int)k < cap; k++)
    {
        out[3 * k] = t[k].mcu_first; out[3 * k + 1] = t[k].info >> 8; out[3 * k + 2] = t[k].row_first;
    }
    *max = (long)b2j::crop_tiles_max(im);
    return (int)n;
}

}
