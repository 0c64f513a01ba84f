// crop_plan.h -- host side of a cropped decode (b2j_batch_set_crops): where a box lies before orientation, and which
// MCUs the IDCT must transform for it. Plain C++, so that the CPU tests check it through tests/native/cropcheck.cpp.
#ifndef B2J_CROP_PLAN_H_INCLUDED
#define B2J_CROP_PLAN_H_INCLUDED

#include <stdint.h>
#include <vector>

#include "b2j_internal.h"

namespace b2j {

// The box (x, y, w, h) of the oriented w x h frame of an image whose scaled, unoriented frame is fw x fh, mapped back to
// that frame through EXIF code `code` (the transform of b2j_batch_set_orientations: codes 5..8 swap the sides). A rectangle
// maps to a rectangle, and orienting the window gives the box. False when the box does not lie inside the oriented frame.
inline bool crop_window(uint32_t fw, uint32_t fh, uint32_t code, const int32_t box[4], CropDev &win)
{
    const bool swap = code >= 5u, mx = code == 2u || code == 3u || code == 7u || code == 8u, my = code == 3u || code == 4u || code == 6u || code == 7u;
    const uint32_t ow = swap ? fh : fw, oh = swap ? fw : fh;
    if (box[0] < 0 || box[1] < 0 || box[2] < 1 || box[3] < 1) return false;
    const uint32_t X = (uint32_t)box[0], Y = (uint32_t)box[1], W = (uint32_t)box[2], H = (uint32_t)box[3];
    if (X >= ow || Y >= oh || W > ow - X || H > oh - Y) return false;
    // destination (X, Y) takes the source pixel (x, y) with (u, v) = (Y, X) for codes 5..8, else (X, Y); x = u or
    // fw - 1 - u (mx); y = v or fh - 1 - v (my)
    const uint32_t u0 = swap ? Y : X, v0 = swap ? X : Y, uw = swap ? H : W, vh = swap ? W : H;
    win.x0 = mx ? fw - u0 - uw : u0;
    win.y0 = my ? fh - v0 - vh : v0;
    win.w = uw;
    win.h = vh;
    return true;
}

// Tiles of the crop tile list of image `img` (descriptor im) for its window `win` at scale `scale`: the MCUs the window
// touches plus `halo` MCUs on each side where the image has them, so that fancy upsampling at the window's edges finds
// its neighbours. An MCU is yh * 8 / scale x yv * 8 / scale output pixels. The MCUs of each MCU row form one run; runs
// that meet (windows as wide as the image) are one run; each run is cut into tiles of at most kTileBlocks / tot_blks
// MCUs. Returns the tiles appended to `out`.
inline uint32_t crop_tiles(const ImgDev &im, uint32_t img, const CropDev &win, uint32_t scale, uint32_t halo, std::vector<TileDev> &out)
{
    const uint32_t mcw = im.mcu_count_w, mch = im.mcu_count / im.mcu_count_w;
    const uint32_t mw = (im.samp & 15u) * 8u / scale, mh = ((im.samp >> 4) & 15u) * 8u / scale;
    const uint32_t c0 = win.x0 / mw, c1 = (win.x0 + win.w - 1u) / mw, r0 = win.y0 / mh, r1 = (win.y0 + win.h - 1u) / mh;
    const uint32_t ca = c0 > halo ? c0 - halo : 0u, cb = c1 + halo < mcw - 1u ? c1 + halo : mcw - 1u;
    const uint32_t ra = r0 > halo ? r0 - halo : 0u, rb = r1 + halo < mch - 1u ? r1 + halo : mch - 1u;
    const uint32_t per_tile = kTileBlocks / im.tot_blks;
    const size_t first = out.size();
    auto emit = [&](uint32_t m, uint32_t end) {
        for (; m < end; m += per_tile)
        {
            const uint32_t n = end - m < per_tile ? end - m : per_tile;
            out.push_back({img, m, im.blk_first + m * im.tot_blks, im.mode | (n << 8)});
        }
    };
    uint32_t run0 = ra * mcw + ca, run1 = run0;   // the open run [run0, run1)
    for (uint32_t r = ra; r <= rb; r++)
    {
        const uint32_t a = r * mcw + ca, b = r * mcw + cb + 1u;
        if (a != run1) { emit(run0, run1); run0 = a; }
        run1 = b;
    }
    emit(run0, run1);
    return (uint32_t)(out.size() - first);
}

// The most tiles crop_tiles() gives for an image, whatever its window and scale: one MCU row's run in tiles, per MCU row.
inline size_t crop_tiles_max(const ImgDev &im)
{
    const uint32_t per_tile = kTileBlocks / im.tot_blks;
    return (size_t)(im.mcu_count / im.mcu_count_w) * ((im.mcu_count_w + per_tile - 1u) / per_tile);
}

} // namespace b2j
#endif
