// kernels.cu -- the sm_100a kernels of the baseline-JPEG decode path and their launchers.
//
//   k_unstuff_fused
//       single-pass pre-pass over the raw entropy-coded bytes: removes byte stuffing and fill bytes, finds the
//       RSTn markers, checks their numbering and emits the start offset of every restart interval
//       in the cleaned stream. Replaces read_more_data<>() (reference decoder.cpp:94-159) and the
//       marker handling of decode_huffman_data() (decoder.cpp:289-307).
//   k_huff_decode
//       one lane per decode segment (restart interval): Huffman decode with shared-memory LUTs,
//       DC prediction, de-zig-zag into a per-lane block staged in shared memory, cooperative
//       128-bit flush of whole 128-byte blocks into the int16 coefficient plane. Replaces
//       decode_huffman_block()/decode_huffman_data() (decoder.cpp:221-365), BitStream's cached
//       reader (bitstream.h:311-365) and HuffmanTree::findCodeInCache() (huffman.h:277-314).
//   k_idct_csc
//       per tile of 192 blocks: coefficient tile staged in swizzled shared memory by a TMA tensor
//       load, thread-per-block dequantise + Chen-Wang IDCT in registers, then chroma
//       replication + exact integer YCbCr->BGRA and 128-bit coalesced stores. Replaces
//       Fast_IDCT (cpuIDCT8x8.cpp:25-127), the upsample/colour loop of decode_mcu_data()
//       (decoder.cpp:429-495) and the OpenCL kernels idct8x8.cl:157-222.
//   k_idct_libjpeg, k_upsample_libjpeg
//       the libjpeg pixel model (B2J_PIXELS_LIBJPEG) instead of k_idct_csc, at every scale (1, 1/2, 1/4, 1/8):
//       libjpeg-turbo's ISLOW or reduced IDCTs into a sample plane, then its chroma upsampling and fixed-point colour.
//   k_idct_gray
//       the libjpeg pixel model in B2J_OUT_GRAY8 (libjpeg's JCS_GRAYSCALE): the luma blocks only, straight into the pixels.
//   k_expand_coefs
//       the reference's coefficient tap (int32, dequantised) from the int16 plane, for parity.
//   k_orient
//       EXIF orientation after the IDCT/colour stage: tiled copies of the images whose code is not 1, rotated or mirrored.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "b2j_internal.h"
#include "b2j_math.h"
#include "b2j_sync.h"
#include "kernels.h"

namespace b2j {

__constant__ uint8_t c_zigzag2[64];   // 2 * natural index of scan position i (byte offset in a block)

static const uint8_t h_zigzag[64] = B2J_ZIGZAG_TABLE;

cudaError_t init_constants()
{
    uint8_t z2[64];
    for (int i = 0; i < 64; i++) z2[i] = (uint8_t)(2 * h_zigzag[i]);
    return cudaMemcpyToSymbol(c_zigzag2, z2, sizeof(z2));
}

// =====================================================================================
// Pre-pass: byte classification.
// For byte b with predecessor p and successor n (all inside one image's scan):
//   b == FF : kept iff n == 00 (stuffed data byte). Otherwise it is a marker prefix / fill byte
//             and is dropped; if n is none of 00, FF, D0..D7 the scan ends here (EOI or any
//             other marker) -- "terminator".
//   b != FF : dropped iff p == FF and b is 00 (stuffing) or D0..D7 (RSTn, recorded as a marker);
//             kept otherwise.
// The reference keeps the Dn byte in its stream and consumes it at the interval switch
// (decoder.cpp:136-141, 296-297); here it is dropped and becomes a segment boundary instead, or, when it starts no
// interval, the end of the data the decoders may read (mark_group).
//
// The classification runs on 4 bytes at a time in a "flag" domain: bit 7 of every byte of a 32-bit
// word is the predicate for that byte (byte j of the thread = bits 8(j&3).. of word j>>2).
struct ScanFlags { uint32_t keep[4], mark[4], term[4]; };

constexpr uint32_t kFlagAll = 0x80808080u;

__device__ __forceinline__ uint32_t eq_ff(uint32_t w)   // flag set where the byte is 0xFF
{
    return ((w & 0x7F7F7F7Fu) + 0x01010101u) & w & kFlagAll;
}
// flags of the first n bytes (n in 0..16) of the thread's 16
__device__ __forceinline__ void first_n_flags(int n, uint32_t m[4])
{
#pragma unroll
    for (int i = 0; i < 4; i++)
    {
        const int r = n - 4 * i;
        m[i] = r >= 4 ? kFlagAll : (r <= 0 ? 0u : (kFlagAll & ((1u << (8 * r)) - 1u)));
    }
}
// 16 flags -> one word with 16 distinct bits (order scrambled; only used for counting / any-tests)
__device__ __forceinline__ uint32_t squeeze(const uint32_t f[4]) { return (f[0] >> 7) | (f[1] >> 6) | (f[2] >> 5) | (f[3] >> 4); }
__device__ __forceinline__ bool flag_at(const uint32_t f[4], int j) { return (f[j >> 2] >> (8 * (j & 3) + 7)) & 1u; }

// The host pads every image's scan with FF D9 D9 ..., so running off the end looks like EOI and no
// end-of-data special case is needed: the pad FF is a terminator and everything behind it is cut
// (bytes behind it, possibly the next image's, are classified too but never used).
// w: the 16 bytes; prev / next: the byte before / after them.
__device__ __forceinline__ ScanFlags classify16(const uint32_t w[4], uint32_t prev, uint32_t next)
{
    ScanFlags f;
    uint32_t F[6], Z[5], D[5];   // index i+1 = word i; F[0] = predecessor, [5] = successor
    F[0] = prev == 0xFFu ? 0x80000000u : 0u;
#pragma unroll
    for (int i = 0; i < 4; i++)
    {
        F[i + 1] = eq_ff(w[i]);
        Z[i] = eq_ff(~w[i]);
        D[i] = eq_ff((w[i] | 0x07070707u) ^ 0x28282828u);   // (b & 0xF8) == 0xD0
    }
    F[5] = next == 0xFFu ? 0x80u : 0u;
    Z[4] = next == 0x00u ? 0x80u : 0u;
    D[4] = (next & 0xF8u) == 0xD0u ? 0x80u : 0u;
#pragma unroll
    for (int i = 0; i < 4; i++)
    {
        const uint32_t Fi = F[i + 1];
        const uint32_t Fp = __funnelshift_l(F[i], Fi, 8);          // flag of the previous byte
        const uint32_t Fn = __funnelshift_r(Fi, F[i + 2], 8);      // flags of the next byte
        const uint32_t Zn = __funnelshift_r(Z[i], Z[i + 1], 8);
        const uint32_t Dn = __funnelshift_r(D[i], D[i + 1], 8);
        f.keep[i] = ((Fi & Zn) | (~Fi & ~(Fp & (Z[i] | D[i])))) & kFlagAll;
        f.mark[i] = ~Fi & Fp & D[i];
        f.term[i] = Fi & ~(Zn | Fn | Dn);
    }
    return f;
}

// A thread's kScanGroups x 16 consecutive bytes of the chunk, loaded with all vector loads in flight
// at once, and their classification. pos = offset of the thread's first byte in the image's scan.
struct ScanThread
{
    uint32_t w[kScanGroups][4];
    ScanFlags f[kScanGroups];

    __device__ __forceinline__ void load_classify(const uint8_t *__restrict__ scan, uint32_t pos)
    {
        uint4 v[kScanGroups];
#pragma unroll
        for (int g = 0; g < kScanGroups; g++) v[g] = __ldg(reinterpret_cast<const uint4 *>(scan + pos) + g);   // 16 B aligned
        const uint32_t prev = pos ? (uint32_t)__ldg(scan + pos - 1) : 0u;
        const uint32_t next = (uint32_t)__ldg(scan + pos + 16 * kScanGroups);                                 // pad bytes exist
#pragma unroll
        for (int g = 0; g < kScanGroups; g++) { w[g][0] = v[g].x; w[g][1] = v[g].y; w[g][2] = v[g].z; w[g][3] = v[g].w; }
#pragma unroll
        for (int g = 0; g < kScanGroups; g++)
            f[g] = classify16(w[g], g ? (w[g - 1][3] >> 24) : prev, g + 1 < kScanGroups ? (w[g + 1][0] & 0xFFu) : next);
    }
    // thread-local position (0 .. 16*kScanGroups-1) of the first terminator, or kNoTerm
    __device__ __forceinline__ uint32_t first_term() const
    {
        uint32_t best = kNoTerm;
#pragma unroll
        for (int g = kScanGroups - 1; g >= 0; g--)
#pragma unroll
            for (int i = 3; i >= 0; i--)
                if (f[g].term[i]) best = 16u * g + 4u * i + ((uint32_t)(__ffs(f[g].term[i]) - 1) >> 3);
        return best;
    }
    // drops the flags of bytes at or behind thread-local position `limit`
    __device__ __forceinline__ void cut(uint32_t limit)
    {
        if (limit >= 16u * kScanGroups) return;
#pragma unroll
        for (int g = 0; g < kScanGroups; g++)
        {
            uint32_t m[4];
            first_n_flags(limit > 16u * g ? (int)min(limit - 16u * g, 16u) : 0, m);
#pragma unroll
            for (int i = 0; i < 4; i++) { f[g].keep[i] &= m[i]; f[g].mark[i] &= m[i]; }
        }
    }
};

// Chunk-local position of the first terminator, or kNoTerm.
__device__ __forceinline__ uint32_t block_first_term(uint32_t local_term, uint32_t tid, uint32_t *s_min)
{
    if (tid == 0) *s_min = kNoTerm;
    __syncthreads();
    if (local_term != kNoTerm) atomicMin(s_min, tid * (16u * kScanGroups) + local_term);
    __syncthreads();
    return *s_min;
}

__device__ __forceinline__ uint32_t local_limit(uint32_t chunk_term, uint32_t tid)
{
    const uint32_t lo = tid * (16u * kScanGroups);
    return chunk_term <= lo ? 0u : chunk_term - lo;   // kNoTerm and anything behind the thread's bytes: no cut
}

// ---- the pre-pass: count, prefix across the chunks of an image and write in ONE kernel.
// Every chunk publishes a 64-bit state word: first its own totals ("aggregate"), later the totals of the
// image up to and including itself ("inclusive"). A chunk obtains its base by looking back over its
// predecessors' words (decoupled look-back: aggregates are added until an inclusive word is met), so no
// chunk waits for more than the local counting of the chunks in front of it, and the bytes are classified
// once instead of twice. CTAs of a grid start in blockIdx order, so a predecessor is always resident or done.
// The word carries everything a successor needs, so relaxed accesses suffice (no fences):
//   bits 63:62 flag (0 empty, 1 aggregate, 2 inclusive) | bit 61 a terminator was met | 60:32 markers | 31:0 kept bytes
// The look-back latency hides behind the compaction: the kept bytes are squeezed into shared memory at their
// CHUNK-LOCAL offsets (which need no base), warp 0 probes its predecessors half-way through its squeezing and
// evaluates the probe afterwards; only the copy-out (shifted to the alignment of the global destination)
// and the restart-interval table wait for the base.
constexpr int kProbeAt = kScanGroups - 1;   // the 16-byte group in front of whose squeeze warp 0 sends its look-back probe
constexpr uint64_t kStAgg = 1ull << 62, kStIncl = 2ull << 62, kStTerm = 1ull << 61;
__device__ __forceinline__ uint64_t st_pack(uint64_t flag, uint32_t keep, uint32_t mark, bool term)
{
    return flag | (term ? kStTerm : 0ull) | ((uint64_t)mark << 32) | keep;
}
__device__ __forceinline__ uint64_t st_load(const uint64_t *p)
{
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_store(uint64_t *p, uint64_t v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Phase A of a 16-byte group: squeeze the dropped bytes out of the registers and store the kept ones to
// shared memory at byte offset o (single bytes up to the next word boundary, whole words, tail bytes).
__device__ __forceinline__ void squeeze_group(uint8_t *__restrict__ s_out, uint32_t o, const uint32_t w[4], const ScanFlags &f, uint32_t nkeep)
{
    uint32_t B[4] = {w[0], w[1], w[2], w[3]};
    if (nkeep != 16u)
    {
        uint32_t keep16 = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) keep16 |= ((((f.keep[i] >> 7) * 0x00204081u) >> 21) & 0xFu) << (4 * i);
        // highest dropped byte first (bytes above the last kept one need no move)
        const uint32_t span = keep16 ? 32u - (uint32_t)__clz(keep16) : 0u;
        uint32_t drop = ~keep16 & ((1u << span) - 1u);
        while (drop)
        {
            const uint32_t j = 31u - (uint32_t)__clz(drop);
            drop ^= 1u << j;
            const uint32_t wi = j >> 2, lm = (1u << (8u * (j & 3u))) - 1u;
            const uint32_t sh0 = __funnelshift_r(B[0], B[1], 8), sh1 = __funnelshift_r(B[1], B[2], 8),
                           sh2 = __funnelshift_r(B[2], B[3], 8), sh3 = B[3] >> 8;
            B[0] = wi == 0u ? ((B[0] & lm) | (sh0 & ~lm)) : B[0];
            B[1] = wi == 1u ? ((B[1] & lm) | (sh1 & ~lm)) : (wi < 1u ? sh1 : B[1]);
            B[2] = wi == 2u ? ((B[2] & lm) | (sh2 & ~lm)) : (wi < 2u ? sh2 : B[2]);
            B[3] = wi == 3u ? ((B[3] & lm) | (sh3 & ~lm)) : sh3;
        }
    }
    uint32_t n = nkeep;
    const uint32_t head = min((4u - (o & 3u)) & 3u, n);
#pragma unroll
    for (int k = 0; k < 3; k++)
        if ((uint32_t)k < head) s_out[o + k] = (uint8_t)(B[0] >> (8 * k));
    if (head)
    {
        const uint32_t hs = head * 8u;   // drop the head bytes from the register array
        B[0] = __funnelshift_r(B[0], B[1], hs);
        B[1] = __funnelshift_r(B[1], B[2], hs);
        B[2] = __funnelshift_r(B[2], B[3], hs);
        B[3] = B[3] >> hs;
    }
    o += head; n -= head;
    uint32_t *wo = reinterpret_cast<uint32_t *>(s_out + o);
#pragma unroll
    for (int k = 0; k < 4; k++)
        if ((uint32_t)(4 * k + 4) <= n) wo[k] = B[k];
    const uint32_t full = n >> 2, tail = n & 3u;
    const uint32_t tw = full == 0u ? B[0] : (full == 1u ? B[1] : (full == 2u ? B[2] : B[3]));
#pragma unroll
    for (int k = 0; k < 3; k++)
        if ((uint32_t)k < tail) s_out[o + full * 4u + k] = (uint8_t)(tw >> (8 * k));
}

// Phase B of a 16-byte group: the restart-interval starts of its RSTn markers (clean_pos = position of the
// group's first kept byte in the image's clean stream, rank = ordinal of the next marker of the image).
// A marker that starts no interval (any RSTn without DRI; the n_segs-th and later ones with DRI) ends the data the
// decoders may read (scan_cut, b2j.h): the reference keeps its Dn byte as data, so a decode past it would differ.
__device__ __forceinline__ void mark_group(const uint32_t w[4], const ScanFlags &f, uint32_t &rank, uint32_t clean_pos, const ImgDev &im,
                                           uint32_t img_idx, uint32_t *__restrict__ seg_start, uint32_t *__restrict__ scan_cut,
                                           int32_t *__restrict__ status)
{
    if (!(f.mark[0] | f.mark[1] | f.mark[2] | f.mark[3])) return;
    uint32_t keep16 = 0, mark16 = 0;
#pragma unroll
    for (int i = 0; i < 4; i++)
    {
        keep16 |= ((((f.keep[i] >> 7) * 0x00204081u) >> 21) & 0xFu) << (4 * i);
        mark16 |= ((((f.mark[i] >> 7) * 0x00204081u) >> 21) & 0xFu) << (4 * i);
    }
    while (mark16)
    {
        const uint32_t j = (uint32_t)__ffs(mark16) - 1u;
        mark16 &= mark16 - 1u;
        const uint32_t at = clean_pos + __popc(keep16 & ((1u << j) - 1u));
        if (im.has_dri && rank + 1 < im.n_segs)
        {
            seg_start[im.seg_first + rank + 1] = at;
            const uint32_t wj = j < 4u ? w[0] : (j < 8u ? w[1] : (j < 12u ? w[2] : w[3]));
            const uint32_t bj = (wj >> (8 * (j & 3u))) & 0xFFu;
            if (bj != 0xD0u + (rank & 7u)) atomicOr(&status[img_idx], B2J_ST_RST_MISMATCH);   // decoder.cpp:298
        }
        else
            atomicMax(&scan_cut[img_idx], ~at);   // zeroed before the decode: the first such marker wins
        rank++;
    }
}

constexpr int kScanMinCtas = 4;   // 64 registers (92 B of spills), 4 CTAs per SM: 0.162 vs 0.164 ms (256 x 1080p), 0.459 vs 0.474 ms (64 x 4K)
__global__ void __launch_bounds__(kScanThreads, kScanMinCtas)
k_unstuff_fused(const uint8_t *__restrict__ raw, uint8_t *__restrict__ clean, const ImgDev *__restrict__ imgs,
                const uint32_t *__restrict__ chunk_img, uint64_t *__restrict__ chunk_state, uint32_t *__restrict__ clean_len,
                uint32_t *__restrict__ seg_start, uint32_t *__restrict__ scan_cut, int32_t *__restrict__ status)
{
    __shared__ uint32_t s_min;
    __shared__ uint32_t s_warp[kScanThreads / 32];
    __shared__ uint32_t s_base[3];   // kept bytes / markers in front of this chunk, dead flag
    __shared__ __align__(16) uint8_t s_out[kScanChunkBytes + 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t c = blockIdx.x;
    const uint32_t img_idx = chunk_img[c];
    const ImgDev &im = imgs[img_idx];
    const uint32_t k = c - im.chunk_first;   // chunk index inside the image
    const uint32_t pos = k * kScanChunkBytes + tid * (16u * kScanGroups);
    ScanThread st;
    st.load_classify(raw + im.raw_off, pos);
    // the scan ends in one chunk per image: only there is the position of the terminator worked out
    uint32_t term = kNoTerm;
    {
        uint32_t any = 0;
#pragma unroll
        for (int g = 0; g < kScanGroups; g++) any |= st.f[g].term[0] | st.f[g].term[1] | st.f[g].term[2] | st.f[g].term[3];
        if (__syncthreads_or(any != 0u))
        {
            term = block_first_term(st.first_term(), tid, &s_min);
            st.cut(local_limit(term, tid));
        }
    }
    uint32_t nkeep[kScanGroups], mine = 0;
#pragma unroll
    for (int g = 0; g < kScanGroups; g++)
    {
        nkeep[g] = __popc(squeeze(st.f[g].keep));
        mine += nkeep[g] | (__popc(squeeze(st.f[g].mark)) << 16);
    }
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += a;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w8 = 0; w8 < kScanThreads / 32; w8++)
    {
        const uint32_t v = s_warp[w8];
        before += (w8 < (int)warp) ? v : 0u;
        total += v;
    }
    const uint32_t own_keep = total & 0xFFFFu, own_mark = total >> 16;
    const bool own_term = term != kNoTerm;
    const uint32_t excl = before + incl - mine;

    // warp 0: publish the aggregate; the (up to 32) nearest predecessors are probed during the squeeze
    uint64_t probe = kStIncl;   // in front of the image: an inclusive zero
    const uint64_t *probe_p = chunk_state + (c - k) + (k - 1u - lane);
    if (warp == 0 && k != 0)
    {
        if (lane == 0) st_store(chunk_state + c, st_pack(kStAgg, own_keep, own_mark, own_term));
    }

    // phase A: squeeze the kept bytes into shared memory at their chunk-local offsets
    {
        uint32_t lo = excl & 0xFFFFu;
#pragma unroll
        for (int g = 0; g < kScanGroups; g++)
        {
            // the probe leaves late in the squeeze (measured: before group 1 / 2 / 3 of 4: 0.167 / 0.164 / 0.162 ms): the neighbouring chunks, which started together with this one,
            // have published their aggregates by then, and the answer is back when the squeeze is finished
            if (g == kProbeAt && warp == 0 && k != 0 && lane < k) probe = st_load(probe_p);
            squeeze_group(s_out, lo, st.w[g], st.f[g], nkeep[g]);
            lo += nkeep[g];
        }
    }

    if (warp == 0)
    {
        uint32_t bk = 0, bm = 0;
        bool dead = false;
        if (k != 0)
        {
            uint32_t j = k;   // predecessors k-1 .. 0 are still to be accounted for
            uint64_t w = probe;
            while (true)
            {
                if (lane < j)
                {
                    // a predecessor publishes its aggregate a few microseconds after it starts; the bound only guards the
                    // GPU against a hang should the in-order start of CTAs ever not hold (flagged, the image is then wrong)
                    uint32_t spins = 0;
                    while ((w >> 62) == 0ull)
                    {
                        if (++spins > (1u << 24)) { atomicOr(&status[img_idx], B2J_ST_INTERNAL); w = kStIncl; break; }
                        w = st_load(probe_p);
                    }
                }
                const uint32_t inc = __ballot_sync(0xFFFFFFFFu, (w >> 62) == 2ull);
                const uint32_t upto = inc ? (uint32_t)__ffs(inc) - 1u : 31u;   // nearest inclusive word (lane order = distance)
                uint32_t kk = lane <= upto ? (uint32_t)w : 0u;
                uint32_t mm = lane <= upto ? (uint32_t)(w >> 32) & 0x1FFFFFFFu : 0u;
                const bool tt = lane <= upto && (w & kStTerm);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { kk += __shfl_xor_sync(0xFFFFFFFFu, kk, o); mm += __shfl_xor_sync(0xFFFFFFFFu, mm, o); }
                bk += kk; bm += mm;
                dead = dead || __any_sync(0xFFFFFFFFu, tt);
                if (inc) break;
                j -= 32u;
                probe_p -= 32;
                w = lane < j ? st_load(probe_p) : kStIncl;
            }
        }
        if (lane == 0)
        {
            // a chunk behind the end of the scan contributes nothing
            st_store(chunk_state + c, dead ? st_pack(kStIncl, bk, bm, true) : st_pack(kStIncl, bk + own_keep, bm + own_mark, own_term));
            s_base[0] = bk; s_base[1] = bm; s_base[2] = dead ? 1u : 0u;
            if (k == 0) seg_start[im.seg_first] = 0;
            if (!dead && (own_term || k + 1u == im.n_chunks))
            {
                // this chunk ends the scan: totals of the image
                clean_len[img_idx] = bk + own_keep;
                // a missing RSTn makes the reference fail with "expected RSTn" (decoder.cpp:298-302)
                if (im.has_dri && bm + own_mark + 1u < im.n_segs) atomicOr(&status[img_idx], B2J_ST_RST_MISMATCH);
            }
        }
    }
    __syncthreads();
    if (s_base[2]) return;   // behind the end of the scan (uniform for the CTA)
    const uint32_t base_keep = s_base[0];

    // phase B: restart-interval table
    {
        uint32_t lo = excl & 0xFFFFu;
        uint32_t rank = s_base[1] + (excl >> 16);   // ordinal of the next RSTn in the image
#pragma unroll
        for (int g = 0; g < kScanGroups; g++)
        {
            mark_group(st.w[g], st.f[g], rank, base_keep + lo, im, img_idx, seg_start, scan_cut, status);
            lo += nkeep[g];
        }
    }
    // copy out: shared byte i goes to clean[g0 + i]. 16-byte vectors at aligned global addresses, assembled
    // from five shared words shifted by the (CTA-uniform) misalignment; single bytes at the two ragged ends.
    const uint64_t g0 = im.raw_off + base_keep;
    const uint32_t a = (uint32_t)(g0 & 15u);
    uint8_t *gd = clean + (g0 - a);                 // aligned; global byte gd[x] <- shared byte x - a
    const uint32_t end = a + own_keep;
    const uint32_t sh = ((4u - (a & 3u)) & 3u) * 8u;
    for (uint32_t v = tid; v * 16u < end; v += kScanThreads)
    {
        const uint32_t lo16 = v * 16u;
        if (lo16 >= a && lo16 + 16u <= end)
        {
            const uint32_t *sw = reinterpret_cast<const uint32_t *>(s_out) + ((lo16 - a) >> 2);
            const uint32_t w0 = sw[0], w1 = sw[1], w2 = sw[2], w3 = sw[3], w4 = sw[4];
            uint4 o;
            o.x = __funnelshift_r(w0, w1, sh); o.y = __funnelshift_r(w1, w2, sh);
            o.z = __funnelshift_r(w2, w3, sh); o.w = __funnelshift_r(w3, w4, sh);
            *reinterpret_cast<uint4 *>(gd + lo16) = o;
        }
        else
        {
            const uint32_t from = lo16 < a ? a : lo16, to = lo16 + 16u < end ? lo16 + 16u : end;
            for (uint32_t q = from; q < to; q++) gd[q] = s_out[q - a];
        }
    }
}

// =====================================================================================
// Huffman decode.
// Per-lane bit reader over the clean stream: a 64-bit big-endian window (cur:nxt) and DEPTH raw words
// of look-ahead. A word is requested DEPTH window shifts before it is needed (it is byte-swapped only
// when it enters the window, so the load itself never blocks). Measured on B200: a 16-byte double-
// buffered queue hides the latency completely but costs more instructions per shift than it saves.
template <int DEPTH>
struct BitReader
{
    uint32_t cur, nxt;     // big-endian words: `cur` holds the bit at `bitpos`
    uint32_t raw[DEPTH];   // look-ahead, memory byte order; raw[0] enters the window next
    uint32_t bitpos;       // 0..31 after refill()
    uint32_t wi;           // index (from wbase) of the next word to fetch: a fixed per-lane base and a 32-bit index
    const uint32_t *wbase; // cost one IMAD.WIDE per fetch; a moving 64-bit pointer costs two more instructions

    // stream: 4-byte aligned base of the image's stream; off: byte offset of the first byte to read
    __device__ __forceinline__ void init(const uint8_t *stream, uint32_t off)
    {
        wbase = reinterpret_cast<const uint32_t *>(stream) + (off >> 2);
        cur = __byte_perm(__ldg(wbase), 0, 0x0123);
        nxt = __byte_perm(__ldg(wbase + 1), 0, 0x0123);
#pragma unroll
        for (int k = 0; k < DEPTH; k++) raw[k] = __ldg(wbase + 2 + k);
        wi = 2 + DEPTH;
        bitpos = (off & 3u) * 8u;
    }
    // words shifted into the window since init()
    __device__ __forceinline__ uint32_t words_fetched() const { return wi - (2u + DEPTH); }
    __device__ __forceinline__ uint32_t peek() const { return __funnelshift_l(nxt, cur, bitpos); }
    __device__ __forceinline__ void refill()
    {
        if (bitpos >= 32u)
        {
            cur = nxt;
            nxt = __byte_perm(raw[0], 0, 0x0123);
#pragma unroll
            for (int k = 0; k + 1 < DEPTH; k++) raw[k] = raw[k + 1];
            raw[DEPTH - 1] = __ldg(wbase + wi);
            wi++;
            bitpos -= 32u;
        }
    }
};

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Shared memory is addressed with explicit 32-bit shared-window addresses in the decode loop: with
// generic pointers the compiler re-derives the window base (S2R SR_CgaCtaId) inside the loop.
__device__ __forceinline__ uint32_t lds_u16(uint32_t a)
{
    uint16_t v;
    asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a)
{
    uint32_t v;
    asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u16(uint32_t a, uint32_t v)
{
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory");
}

// One symbol from a two-level LUT in shared memory (entry format: b2j_internal.h). `tab` is the
// shared-window byte address of the table. Returns the leaf entry, 0 when no codeword matches.
__device__ __forceinline__ uint32_t lut_first(uint32_t tab, uint32_t pk, uint32_t bits = kLutBits)
{
    return lds_u16(tab + ((pk >> (32u - bits)) << 1));
}
// Second level, taken when bit 5 of the first-level entry is clear (bit 5 is set in every leaf:
// 32 + len). Returns a leaf, or 0 when the bits are no codeword.
__device__ __forceinline__ uint32_t lut_second(uint32_t tab, uint32_t pk, uint32_t e, uint32_t bits = kLutBits)
{
    if (e != 0u)
    {
        const uint32_t nb = e & 63u, off = (e >> 6) * kLutSubAlign;
        e = lds_u16(tab + (((1u << bits) + off + ((pk << bits) >> (32u - nb))) << 1));
    }
    return e;
}

// Value bits -> signed coefficient (JPEG EXTEND, decoder.cpp:72-82). v: the bits left-aligned, size = their
// number (0 -> 0). A leading 1 bit means positive.
__device__ __forceinline__ int32_t extend_sz(uint32_t v, uint32_t size)
{
    const uint32_t u = __funnelshift_l(v, 0u, size);                 // the value bits as a number: v >> (32 - size)
    const uint32_t neg = (uint32_t)((int32_t)~v >> 31);              // all ones when the leading bit is 0
    return (int32_t)(u - __funnelshift_l(neg, 0u, size));            // negative: u - (2^size - 1)
}

// Clean bytes of an image the decoders may read: its clean stream, up to the first restart marker that starts no
// interval (mark_group; scan_cut holds its complement, 0 = none). Reading past the end flags B2J_ST_OVERRUN.
__device__ __forceinline__ uint32_t stream_len(const uint32_t *__restrict__ clean_len, const uint32_t *__restrict__ scan_cut, uint32_t img)
{
    return min(clean_len[img], ~scan_cut[img]);
}

// SYNC = false: a lane is a restart interval (byte-aligned start from seg_start[], DC predictors 0, the
//   block-in-MCU phase is 0 and therefore uniform across the warp).
// SYNC = true : a lane is a sub-sequence of a stream without restart markers; its first block, bit
//   position, MCU phase, block index and DC predictors come from the self-synchronisation passes
//   (SubRec / SubPre), and the table choice is per lane.
constexpr uint32_t kZzBytes = 192;   // 128 zig-zag offsets + 64 bytes of scratch for the CTA-wide prefix of the SYNC lanes
template <bool SYNC>
__global__ void __launch_bounds__(kHuffThreads)
k_huff_decode(const uint8_t *__restrict__ clean, const ImgDev *__restrict__ imgs, const HuffCtaDev *__restrict__ ctas,
              const uint32_t *__restrict__ seg_start, const uint32_t *__restrict__ clean_len, const uint32_t *__restrict__ scan_cut,
              const uint16_t *__restrict__ luts, int16_t *__restrict__ coef, int32_t *__restrict__ status,
              const SubRec *__restrict__ recs, const uint4 *__restrict__ cta_base)
{
    extern __shared__ __align__(16) uint8_t smem[];
    // [ per-lane block slots: kHuffThreads * 128 B ][ zig-zag byte offsets: 64 B ][ LUT set ]
    uint8_t *s_slots = smem;
    uint8_t *s_zz2 = smem + kHuffThreads * 128;                 // lanes sit at different scan positions: shared, not constant, memory;
                                                                // 128 entries: a corrupt block may run up to 15 positions past 63
    uint16_t *s_lut = reinterpret_cast<uint16_t *>(smem + kHuffThreads * 128 + kZzBytes);

    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const HuffCtaDev cta = ctas[blockIdx.x];
    const ImgDev &im = imgs[cta.img];

    // stage the LUT set (16-byte granules) and clear the slots
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(luts + im.lut_off);
        uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
        for (uint32_t k = tid; k < im.lut_dec_len / 8; k += kHuffThreads) dst[k] = __ldg(src + k);
        uint4 *z = reinterpret_cast<uint4 *>(s_slots);
        for (uint32_t k = tid; k < kHuffThreads * 8; k += kHuffThreads) z[k] = make_uint4(0, 0, 0, 0);
        if (tid < 128) s_zz2[tid] = tid < 64 ? c_zigzag2[tid] : (uint8_t)0;
    }
    __syncthreads();

    const uint32_t tot = im.tot_blks, ny = im.ny_blks, nyu = im.ny_blks + im.nu_blks;
    const uint32_t seg = cta.seg_first + tid;
    uint32_t start = 0, end = 0, nblk = 0, blk0 = 0, start_bit = 0, bi = 0;
    int32_t dc0 = 0, dc1 = 0, dc2 = 0;
    int32_t err = 0;
    bool check_end = false, active, decodable;
    if (!SYNC)
    {
        active = seg < im.n_segs;
        if (active)
        {
            start = seg_start[im.seg_first + seg];
            const uint32_t mcu0 = seg * im.restart_interval;
            const uint32_t nmcu = min(im.restart_interval, im.mcu_count - mcu0);
            nblk = nmcu * tot;
            blk0 = im.blk_first + mcu0 * tot;
            if (seg + 1 < im.n_segs) { end = seg_start[im.seg_first + seg + 1]; check_end = (end != kSegInvalid); }
            if (!check_end) end = stream_len(clean_len, scan_cut, cta.img);
        }
        // a lane whose start is unknown (missing RSTn) still emits zero blocks so the plane is defined
        decodable = active && start != kSegInvalid;
    }
    else
    {
        const uint32_t bits = stream_len(clean_len, scan_cut, cta.img) * 8u;
        const uint32_t n_sub = (bits + kSubBytes * 8 - 1) / (kSubBytes * 8);
        active = seg < n_sub && tid < (uint32_t)kSyncLanes;   // a decode CTA covers one chunk of the synchronisation
        SubRec rec;
        rec.nblk = 0; rec.dc[0] = rec.dc[1] = rec.dc[2] = 0;
        if (active) rec = recs[im.sub_first + seg];
        // exclusive prefix of (blocks started, DC sums) over the sub-sequences in front of this lane: the CTA's base
        // (k_sync_cta_scan) plus the lanes in front of it inside the CTA
        SubPre pre;
        {
            uint4 *s_wtot = reinterpret_cast<uint4 *>(smem + kHuffThreads * 128 + 128);   // static shared memory would misalign the slots
            uint32_t ib = rec.nblk; int32_t i0 = rec.dc[0], i1 = rec.dc[1], i2 = rec.dc[2];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const uint32_t tb = __shfl_up_sync(0xFFFFFFFFu, ib, o);
                const int32_t t0 = __shfl_up_sync(0xFFFFFFFFu, i0, o), t1 = __shfl_up_sync(0xFFFFFFFFu, i1, o), t2 = __shfl_up_sync(0xFFFFFFFFu, i2, o);
                if (lane >= (uint32_t)o) { ib += tb; i0 += t0; i1 += t1; i2 += t2; }
            }
            if (lane == 31u) s_wtot[tid >> 5] = make_uint4(ib, (uint32_t)i0, (uint32_t)i1, (uint32_t)i2);
            __syncthreads();
            uint4 acc = cta_base[blockIdx.x];
#pragma unroll
            for (int w = 0; w < kHuffThreads / 32; w++)
                if (w < (int)(tid >> 5)) { const uint4 t = s_wtot[w]; acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w; }
            pre.blk = acc.x + ib - rec.nblk;
            pre.dc[0] = (int32_t)acc.y + i0 - rec.dc[0]; pre.dc[1] = (int32_t)acc.z + i1 - rec.dc[1]; pre.dc[2] = (int32_t)acc.w + i2 - rec.dc[2];
        }
        if (active && rec.fs != kSubNone && pre.blk < im.blk_count)
        {
            nblk = min(rec.nblk, im.blk_count - pre.blk);           // bits behind the last block decode to junk blocks: dropped
            blk0 = im.blk_first + pre.blk;
            start_bit = rec.fs;
            bi = rec.fc;
            dc0 = pre.dc[0]; dc1 = pre.dc[1]; dc2 = pre.dc[2];
        }
        // the stream ends before the last block (an empty stream has no sub-sequence: lane 0 of the first CTA reports it)
        if (tid < (uint32_t)kSyncLanes && seg + 1 == max(n_sub, 1u) && pre.blk + rec.nblk < im.blk_count) err |= B2J_ST_OVERRUN;
        decodable = active && nblk > 0;
        // Lanes change places: sorted by the phase of their first block inside the MCU, then by falling block count.
        // The decode loop below runs block by block in warp lockstep, so a warp costs (longest lane in blocks) x
        // (longest block of every round): lanes of one phase meet the same component in every round, and neighbours
        // in block count finish together. Counting sort over 640 keys in the (still zero) slot area.
        {
            uint32_t *s_hist = reinterpret_cast<uint32_t *>(s_slots);      // [640] counters, then their exclusive prefix
            uint32_t *s_wsum = s_hist + 640;                               // [4] warp totals of the scan
            uint32_t *s_desc = s_hist + 648;                               // [kHuffThreads][6] work descriptors
            const uint32_t key = decodable ? bi * 64u + (63u - min(nblk, 63u)) : 639u;
            const uint32_t within = atomicAdd(&s_hist[key], 1u);
            __syncthreads();
            uint32_t h[5], sum = 0;
#pragma unroll
            for (int k = 0; k < 5; k++) { h[k] = s_hist[tid * 5u + k]; sum += h[k]; }
            uint32_t inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                if (lane >= (uint32_t)o) inc += t;
            }
            if (lane == 31u) s_wsum[tid >> 5] = inc;
            __syncthreads();
            uint32_t run = inc - sum;
#pragma unroll
            for (int w = 0; w < kHuffThreads / 32; w++) run += (w < (int)(tid >> 5)) ? s_wsum[w] : 0u;
#pragma unroll
            for (int k = 0; k < 5; k++) { s_hist[tid * 5u + k] = run; run += h[k]; }
            __syncthreads();
            uint32_t *d = s_desc + (s_hist[key] + within) * 6u;
            d[0] = nblk | bi << 16; d[1] = blk0; d[2] = start_bit; d[3] = (uint32_t)dc0; d[4] = (uint32_t)dc1; d[5] = (uint32_t)dc2;
            __syncthreads();
            const uint32_t *m = s_desc + tid * 6u;
            nblk = m[0] & 0xFFFFu; bi = m[0] >> 16; blk0 = m[1]; start_bit = m[2];
            dc0 = (int32_t)m[3]; dc1 = (int32_t)m[4]; dc2 = (int32_t)m[5];
            decodable = nblk > 0;
            end = bits >> 3;   // every lane may hold work now, whatever its own sub-sequence was
            __syncthreads();
            uint4 *z = reinterpret_cast<uint4 *>(s_slots);
            for (uint32_t k = tid; k < (648u + kHuffThreads * 6u + 3u) / 4u; k += kHuffThreads) z[k] = make_uint4(0, 0, 0, 0);
            __syncthreads();
        }
        start = start_bit >> 3;
    }

    BitReader<1> br;
    br.init(clean + im.raw_off, decodable ? start : 0u);
    const uint32_t bit0 = br.bitpos;          // consumed bits are counted from byte `start`
    const uint32_t seg_bytes = end > start ? end - start : 0u;   // !SYNC: what the lane may consume
    if (SYNC) br.bitpos += start_bit & 7u;
    bool dead = !decodable;

    uint32_t sm_base;   // kept opaque: otherwise the shared-window base is re-derived (S2R) inside the decode loop
    asm volatile("mov.u32 %0, %1;" : "=r"(sm_base) : "r"(smem_addr(smem)));
    const uint32_t sm_zz = sm_base + kHuffThreads * 128;
    const uint32_t sm_lut = sm_zz + kZzBytes;
    // shared address of this lane's slot with the chunk swizzle folded in: coefficient n lives at
    // slot + ((n>>3) ^ (lane&7))*16 + (n&7)*2 == slot_key ^ (2n)   (slots are 128-byte aligned)
    const uint32_t slot_key = sm_base + tid * 128u + ((lane & 7u) << 4);

    const uint32_t max_nblk = __reduce_max_sync(0xFFFFFFFFu, nblk);
    // bi: block index inside the MCU (!SYNC: uniform across the warp, segments start on MCU boundaries)
    for (uint32_t b = 0; b < max_nblk; b++)
    {
        const uint32_t comp = (bi >= ny ? 1u : 0u) + (bi >= nyu ? 1u : 0u);
        const uint32_t dc_tab = sm_lut + 2u * (uint32_t)s_lut[comp];
        const uint32_t ac_tab = sm_lut + 2u * (uint32_t)s_lut[3 + comp];
        const bool mine = b < nblk;
        if (mine && !dead)
        {
            // ---- DC (decoder.cpp:226-233)
            uint32_t pk = br.peek();
            uint32_t e = lut_first(dc_tab, pk, kLutBitsDc);
            if (!(e & 32u)) e = lut_second(dc_tab, pk, e, kLutBitsDc);
            if (!(e & 32u)) { err |= B2J_ST_BAD_CODE; dead = true; }
            else
            {
                uint32_t len = e & 31u, size = (e >> 6) & 31u;
                const int32_t diff = extend_sz(pk << len, size);
                br.bitpos += len + size;
                br.refill();
                int32_t dcv;
                if (comp == 0) { dc0 += diff; dcv = dc0; }
                else if (comp == 1) { dc1 += diff; dcv = dc1; }
                else { dc2 += diff; dcv = dc2; }
                if (dcv != (int32_t)(int16_t)dcv) err |= B2J_ST_DC_RANGE;
                sts_u16(slot_key, (uint32_t)dcv);
                // ---- AC (decoder.cpp:236-258). The end-of-block code carries a run of 63 in the table, so it
                // leaves the loop through the ordinary position test and costs no test of its own.
                uint32_t pos = 1;
                while (true)
                {
                            pk = br.peek();
                    e = lut_first(ac_tab, pk);
                    if (!(e & 32u))
                    {
                        e = lut_second(ac_tab, pk, e);
                        if (!(e & 32u)) { err |= B2J_ST_BAD_CODE; dead = true; break; }
                    }
                    len = e & 31u;
                    size = (e >> 6) & 15u;
                    const int32_t v = extend_sz(pk << len, size);
                    br.bitpos += len + size;
                    br.refill();
                    pos += e >> 10;          // zero run
                    if (size) sts_u16(slot_key ^ lds_u8(sm_zz + pos), (uint32_t)v);   // pos < 128: the table is padded
                    pos++;   // past the stored coefficient, or the extra zero of a size-0 run (decoder.cpp:247-252)
                    if (pos >= 64u) break;
                }
                // more than 64 coefficients without an end-of-block code (decoder.cpp:259)
                if (!dead && pos > 64u && (e >> 10) != kRunEob) { err |= B2J_ST_BLOCK_OVERFLOW; dead = true; }
            }
        }
        __syncwarp();
        // ---- cooperative flush: 8 lanes move one 128-byte block, 4 blocks per step
        const uint32_t my_dst = mine ? (blk0 + b) : 0xFFFFFFFFu;
        const uint32_t warp_slot0 = (tid & ~31u) * 128u;
#pragma unroll
        for (int it = 0; it < 8; it++)
        {
            const uint32_t j = (uint32_t)it * 4u + (lane >> 3);   // source lane
            const uint32_t dst = __shfl_sync(0xFFFFFFFFu, my_dst, j);
            const uint32_t ch = lane & 7u;
            if (dst != 0xFFFFFFFFu)
            {
                uint4 *sp = reinterpret_cast<uint4 *>(s_slots + warp_slot0 + j * 128u + ((ch ^ (j & 7u)) << 4));
                const uint4 v = *sp;
                *sp = make_uint4(0, 0, 0, 0);
                *reinterpret_cast<uint4 *>(coef + (size_t)dst * 64 + ch * 8) = v;
            }
        }
        __syncwarp();
        // A lane whose segment is truncated or corrupt must not keep reading whatever follows it (other images,
        // the scratch arrays, the end of the allocation): once it has fetched more than its segment holds, plus the
        // reader's look-ahead, it stops and the image is flagged (decoder.cpp:310-314 "data incomplete").
        if (!SYNC && !dead)
        {
            const uint32_t nw_now = br.words_fetched();
            if (nw_now * 4u > seg_bytes + 16u) { err |= B2J_ST_OVERRUN; dead = true; }
        }
        bi = (bi + 1 == tot) ? 0u : bi + 1;
    }

    if (decodable && !dead)
    {
        // bits consumed since `start`; a restart interval must end exactly at its marker
        // (decoder.cpp:296-302 aligns to the byte boundary and expects RSTn there)
        const uint32_t nw = br.words_fetched();
        const uint64_t bits = (uint64_t)nw * 32u + br.bitpos - bit0;
        const uint64_t used = (bits + 7u) >> 3;
        const uint64_t avail = (uint64_t)end - start;
        if (used > avail) err |= B2J_ST_OVERRUN;
        else if (!SYNC && check_end && used != avail) err |= B2J_ST_SEGMENT_END;
    }
    if (err) atomicOr(&status[cta.img], err);
}

// =====================================================================================
// Self-synchronising entropy decode for streams without restart markers (north_star (1)).
//
// The clean stream of an image is cut into sub-sequences of kSubBytes*8 bits, one lane each. A JPEG
// decoder state is (bit position, block index inside the MCU, zig-zag position); Huffman codes
// self-synchronise, so a lane that starts from a GUESSED state at its sub-sequence border usually
// falls into step with the true decoder within a few dozen symbols. Kernels:
//   k_sync_chunks   one CTA per chunk of kSyncLanes sub-sequences: round 0 and all further rounds of the chunk in
//                   shared memory (b2j_sync.h), records + chunk totals + chunk entry/exit state out;
//   k_sync_sweep    one CTA per image: every chunk must have started from its predecessor's exit state; the rare
//                   chunk that did not is repaired, in order: one thread walks its sub-sequences again from the
//                   true entry state until a walk falls into step with the old records -- correctness does not
//                   depend on luck;
//   k_sync_cta_scan exclusive prefix of block counts and DC sums over the chunks -> first block index and DC
//                   predictors of every chunk;
//   k_huff_decode<SYNC>  every lane decodes the blocks that START in its sub-sequence.
// The walk itself (walk_stream) lives in b2j_sync.h, shared with the host emulation. Device view of the tables:
// the LUT set staged in shared memory, addressed through the 32-bit shared window.
struct DevLut
{
    uint32_t sm;            // shared-window byte address of the WALK part of the set (what the sync kernels stage)
    uint32_t walk0;         // u16 offset of the walk part inside the set
    uint32_t ct;            // shared-window byte address of the per-block table (WalkCtab[16])
    const uint16_t *g;      // the whole set in global memory: header and decode tables (the rare one-symbol path)
    __device__ __forceinline__ uint32_t at(uint32_t i) const { return __ldg(g + i); }
    __device__ __forceinline__ uint32_t tab(uint32_t off16) const { return sm + ((off16 - walk0) << 1); }
    __device__ __forceinline__ uint32_t ld(uint32_t h, uint32_t i) const { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(h + (i << 2))); return v; }
    __device__ __forceinline__ WalkCtab ctab(uint32_t c) const
    {
        WalkCtab t;
        const uint32_t a = ct + c * (uint32_t)sizeof(WalkCtab);
        asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(t.tdc), "=r"(t.tac), "=r"(t.next), "=r"(t.comp) : "r"(a));
        asm("ld.shared.v2.u32 {%0, %1}, [%2+16];" : "=r"(t.m1), "=r"(t.m2) : "r"(a));
        t.pad0 = t.pad1 = 0u;
        return t;
    }
    __device__ __forceinline__ uint32_t hdr(int i) const { return __ldg(g + i); }
};

struct DevWalk
{
    StreamWords stream;
    DevLut lut;
    // s_ctab: 16 WalkCtab of shared memory, filled here by the first `tot` threads (the caller synchronises afterwards)
    __device__ __forceinline__ void init(const uint8_t *clean_img, uint32_t sm_walk, const uint16_t *g_lut, WalkCtab *s_ctab, const ImgDev &im)
    {
        stream.w = reinterpret_cast<const uint32_t *>(clean_img);
        lut.sm = sm_walk; lut.g = g_lut; lut.walk0 = im.lut_dec_len;
        asm volatile("mov.u32 %0, %1;" : "=r"(lut.ct) : "r"(smem_addr(s_ctab)));   // opaque: otherwise the window base is re-derived inside the loop
        if (threadIdx.x < im.tot_blks && threadIdx.x < 16u) s_ctab[threadIdx.x] = walk_ctab_entry(lut, threadIdx.x, im.ny_blks, im.nu_blks, im.tot_blks);
    }
    __device__ __forceinline__ WalkResult walk(WalkState s, uint32_t limit) const { return walk_stream(stream, lut, s, limit); }
};

// ---- chunk-wise synchronisation (b2j_sync.h): all rounds of a chunk of kSyncLanes sub-sequences inside one CTA.
// Shared memory: [ SyncShared ][ LUT set ].
constexpr uint32_t kSyncSharedBytes = (sizeof(SyncShared) + 15u) & ~15u;

// Runs one chunk (round 0, the rounds, output). All threads of the CTA; `wk` walks this image's stream.
// chunk_state[k] = (entry state assumed for the first lane, exit state of the last lane); cta_tot[k] = totals of the chunk.
__device__ __forceinline__ void sync_run_chunk(const DevWalk &wk, SyncShared &sh, const SyncChunk &ch, SubRec *__restrict__ rec_img,
                                               uint4 *chunk_state_k, uint4 *cta_tot_k, uint32_t *__restrict__ stats, uint4 *s_wtot)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    sync_phase_round0(wk, ch, sh, tid);
    __syncthreads();
    for (uint32_t round = 1; round <= (uint32_t)kHuffThreads + 1u; round++)   // lane k of a chunk is final after k rounds
    {
        if (tid == 0) sh.nq = 0u;
        uint2 entry;
        const bool need = sync_phase_need(ch, sh, tid, entry);
        if (!__syncthreads_or(need)) break;   // also orders the reads of cur[] above before the writes below
        bool met = true;
        if (need)
        {
            met = sync_lane_first(wk, ch, sh, tid, entry, false);
            if (!met) sh.q[atomicAdd(&sh.nq, 1u)] = (uint8_t)tid;
        }
        const int missed = __syncthreads_count(need && !met);
        // the lanes that did not meet their checkpoint, packed into the first warps
        if (tid < (uint32_t)missed) sync_lane_second(wk, ch, sh, sh.q[tid], false);
        if (tid == 0 && missed && stats) atomicAdd(&stats[round < 6u ? round : 6u], (uint32_t)missed);
        __syncthreads();
    }
    // ---- output: the records of the chunk's own lanes, its totals, its entry and exit state
    const bool out = tid >= (uint32_t)kSyncPre && sync_lane_active(ch, tid);
    uint32_t nb = 0; int32_t d0 = 0, d1 = 0, d2 = 0;
    if (out)
    {
        const SubRec c = sh.cur[tid];
        uint4 a, b;
        a.x = c.p; a.y = c.cz; a.z = c.nblk; a.w = (uint32_t)c.dc[0];
        b.x = (uint32_t)c.dc[1]; b.y = (uint32_t)c.dc[2]; b.z = c.fs; b.w = c.fc;
        uint4 *dst = reinterpret_cast<uint4 *>(rec_img + sync_lane_sub(ch, tid));
        dst[0] = a; dst[1] = b;
        nb = c.nblk; d0 = c.dc[0]; d1 = c.dc[1]; d2 = c.dc[2];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        nb += __shfl_xor_sync(0xFFFFFFFFu, nb, o); d0 += __shfl_xor_sync(0xFFFFFFFFu, d0, o);
        d1 += __shfl_xor_sync(0xFFFFFFFFu, d1, o); d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, o);
    }
    if (lane == 0) s_wtot[tid >> 5] = make_uint4(nb, (uint32_t)d0, (uint32_t)d1, (uint32_t)d2);
    __syncthreads();
    if (tid == 0)
    {
        uint4 t = s_wtot[0];
#pragma unroll
        for (int w = 1; w < kHuffThreads / 32; w++) { t.x += s_wtot[w].x; t.y += s_wtot[w].y; t.z += s_wtot[w].z; t.w += s_wtot[w].w; }
        *cta_tot_k = t;
        const uint32_t n_out = min((uint32_t)kSyncLanes, ch.n_sub - ch.first);
        const uint32_t last = (uint32_t)kSyncPre + n_out - 1u;
        *chunk_state_k = make_uint4(sh.entry_used[kSyncPre].x, sh.entry_used[kSyncPre].y, sh.cur[last].p, sh.cur[last].cz);
    }
    __syncthreads();   // s_wtot and sh may be reused by the caller
}

// The walk part of the image's LUT set (the walk tables; the decode part stays in global memory) into shared memory.
__device__ __forceinline__ void sync_stage_lut(uint16_t *s_lut, const uint16_t *__restrict__ luts, const ImgDev &im)
{
    const uint4 *src = reinterpret_cast<const uint4 *>(luts + im.lut_off + im.lut_dec_len);
    uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
    for (uint32_t k = threadIdx.x; k < (im.lut_len - im.lut_dec_len) / 8; k += kHuffThreads) dst[k] = __ldg(src + k);
}

// One CTA per chunk. use_pre: walk kSyncPre sub-sequences in front of the chunk to find its entry state (0: every chunk
// but the first starts from the bare guess, so that every border is repaired by the sweep -- a test knob).
__global__ void __launch_bounds__(kHuffThreads)
k_sync_chunks(const uint8_t *__restrict__ clean, const ImgDev *__restrict__ imgs, const HuffCtaDev *__restrict__ ctas,
              const uint32_t *__restrict__ clean_len, const uint32_t *__restrict__ scan_cut, const uint16_t *__restrict__ luts,
              SubRec *__restrict__ recs, uint4 *__restrict__ chunk_state, uint4 *__restrict__ cta_tot, uint32_t *__restrict__ stats, uint32_t use_pre)
{
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ uint4 s_wtot[kHuffThreads / 32];
    __shared__ __align__(16) WalkCtab s_ctab[16];
    SyncShared &sh = *reinterpret_cast<SyncShared *>(smem);
    uint16_t *s_lut = reinterpret_cast<uint16_t *>(smem + kSyncSharedBytes);
    const HuffCtaDev cta = ctas[blockIdx.x];
    const ImgDev &im = imgs[cta.img];
    const uint32_t bits = stream_len(clean_len, scan_cut, cta.img) * 8u;
    const uint32_t n_sub = (bits + kSubBytes * 8 - 1) / (kSubBytes * 8);
    if (cta.seg_first >= n_sub)
    {
        // uniform: the clean stream is shorter than the raw bound; the chunk contributes nothing
        if (threadIdx.x == 0) { cta_tot[blockIdx.x] = make_uint4(0u, 0u, 0u, 0u); chunk_state[blockIdx.x] = make_uint4(0u, 0u, 0u, 0u); }
        return;
    }
    sync_stage_lut(s_lut, luts, im);
    __syncthreads();
    uint32_t sm_lut;
    asm volatile("mov.u32 %0, %1;" : "=r"(sm_lut) : "r"(smem_addr(smem) + kSyncSharedBytes));
    DevWalk wk;
    wk.init(clean + im.raw_off, sm_lut, luts + im.lut_off, s_ctab, im);
    __syncthreads();
    SyncChunk ch;
    ch.first = cta.seg_first; ch.n_sub = n_sub; ch.bits = bits;
    const bool pre = use_pre != 0u && cta.seg_first != 0u;
    ch.first_lane = pre ? (cta.seg_first >= (uint32_t)kSyncPre ? 0u : (uint32_t)kSyncPre - cta.seg_first) : (uint32_t)kSyncPre;
    ch.forced = cta.seg_first == 0u;          // the first chunk of an image starts from the true state
    ch.forced_entry = make_uint2(0u, 0u);
    sync_run_chunk(wk, sh, ch, recs + im.sub_first, chunk_state + blockIdx.x, cta_tot + blockIdx.x, stats, s_wtot);
}

// One CTA per image: every chunk must have started from the state its predecessor ended in. All threads compare; the
// first chunk that does not is repaired by one thread (sync_repair_chunk), then the search goes on behind it (its exit state
// may have changed). With pre-lanes this finds nothing in almost every image and costs one pass over the chunk states.
__global__ void __launch_bounds__(kHuffThreads)
k_sync_sweep(const uint8_t *__restrict__ clean, const ImgDev *__restrict__ imgs, const uint32_t *__restrict__ sync_imgs,
             const uint32_t *__restrict__ clean_len, const uint32_t *__restrict__ scan_cut, const uint16_t *__restrict__ luts,
             SubRec *__restrict__ recs, uint4 *chunk_state, uint4 *cta_tot, uint32_t *__restrict__ stats)
{
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ __align__(16) WalkCtab s_ctab[16];
    __shared__ uint32_t s_min;
    uint16_t *s_lut = reinterpret_cast<uint16_t *>(smem + kSyncSharedBytes);
    const uint32_t tid = threadIdx.x;
    const uint32_t img = sync_imgs[blockIdx.x];
    const ImgDev &im = imgs[img];
    const uint32_t bits = stream_len(clean_len, scan_cut, img) * 8u;
    const uint32_t n_sub = (bits + kSubBytes * 8 - 1) / (kSubBytes * 8);
    const uint32_t nc = (n_sub + (uint32_t)kSyncLanes - 1u) / (uint32_t)kSyncLanes;
    uint4 *state = chunk_state + im.scta_first;
    uint4 *tot = cta_tot + im.scta_first;
    bool lut_ready = false;
    uint32_t c_start = 1u, repaired = 0u;
    while (c_start < nc)
    {
        // the first chunk at or behind c_start whose entry state is not its predecessor's exit state
        uint32_t found = nc;
        for (uint32_t base = c_start; base < nc; base += kHuffThreads)
        {
            const uint32_t c = base + tid;
            bool bad = false;
            if (c < nc)
            {
                const uint4 mine = __ldcg(state + c), prev = __ldcg(state + c - 1u);
                bad = mine.x != prev.z || mine.y != prev.w;
            }
            if (!__syncthreads_or(bad)) continue;
            if (tid == 0) s_min = nc;
            __syncthreads();
            if (bad) atomicMin(&s_min, c);
            __syncthreads();
            found = s_min;
            break;
        }
        if (found >= nc) break;
        if (!lut_ready)
        {
            sync_stage_lut(s_lut, luts, im);
            lut_ready = true;
        }
        __syncthreads();
        uint32_t sm_lut;
        asm volatile("mov.u32 %0, %1;" : "=r"(sm_lut) : "r"(smem_addr(smem) + kSyncSharedBytes));
        DevWalk wk;
        wk.init(clean + im.raw_off, sm_lut, luts + im.lut_off, s_ctab, im);
        __syncthreads();
        if (tid == 0)
        {
            // one thread chases the change downstream; nearly always the first walk already falls into step
            const uint4 prev = __ldcg(state + found - 1u), mine = __ldcg(state + found);
            const uint4 t = __ldcg(tot + found);
            uint32_t t4[4] = {t.x, t.y, t.z, t.w};
            uint2 exit_pcz = make_uint2(mine.z, mine.w);
            sync_repair_chunk(wk, found, n_sub, bits, recs + im.sub_first, make_uint2(prev.z, prev.w), t4, exit_pcz);
            __stcg(tot + found, make_uint4(t4[0], t4[1], t4[2], t4[3]));
            __stcg(state + found, make_uint4(prev.z, prev.w, exit_pcz.x, exit_pcz.y));
        }
        __threadfence_block();
        __syncthreads();
        repaired++;
        c_start = found + 1u;
    }
    if (tid == 0 && repaired) atomicAdd(&stats[7], repaired);   // chunks whose pre-lanes had not fallen into step
}

// One warp per image: exclusive scan of its CTA totals (in place: totals in, bases out).
__global__ void __launch_bounds__(32)
k_sync_cta_scan(const ImgDev *__restrict__ imgs, const uint32_t *__restrict__ sync_imgs, uint4 *__restrict__ cta_tot)
{
    const uint32_t lane = threadIdx.x;
    const ImgDev &im = imgs[sync_imgs[blockIdx.x]];
    const uint32_t n = (im.n_sub_max + (uint32_t)kSyncLanes - 1u) / (uint32_t)kSyncLanes;
    uint4 *t = cta_tot + im.scta_first;
    uint4 run = make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t b0 = 0; b0 < n; b0 += 32u)
    {
        const uint32_t k = b0 + lane;
        const uint4 v = k < n ? t[k] : make_uint4(0u, 0u, 0u, 0u);
        uint4 x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, x.x, o), b = __shfl_up_sync(0xFFFFFFFFu, x.y, o),
                           c = __shfl_up_sync(0xFFFFFFFFu, x.z, o), d = __shfl_up_sync(0xFFFFFFFFu, x.w, o);
            if (lane >= (uint32_t)o) { x.x += a; x.y += b; x.z += c; x.w += d; }
        }
        if (k < n) t[k] = make_uint4(run.x + x.x - v.x, run.y + x.y - v.y, run.z + x.z - v.z, run.w + x.w - v.w);
        run.x += __shfl_sync(0xFFFFFFFFu, x.x, 31); run.y += __shfl_sync(0xFFFFFFFFu, x.y, 31);
        run.z += __shfl_sync(0xFFFFFFFFu, x.z, 31); run.w += __shfl_sync(0xFFFFFFFFu, x.w, 31);
    }
}

// =====================================================================================
// IDCT + upsample + colour.
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_addr(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(smem_addr(bar)) : "memory");
}

// Packed clamp(a + b, 0, 255) on two int16 lanes.
__device__ __forceinline__ uint32_t addclamp2(uint32_t a, uint32_t b)
{
    return __viaddmin_s16x2_relu(a, b, 0x00FF00FFu);
}

// Two column-pass outputs that already carry the +256 bias -> one word of two unsigned 16-bit samples
// clipped to [0, 511], i.e. the reference's clip to [-256, 255] (cpuIDCT8x8.cpp:13-23): the pack
// saturates below 0 (and above 65535), the packed min cuts at 511.
__device__ __forceinline__ uint32_t pack_clip2(int32_t lo, int32_t hi)
{
    uint32_t d;
    asm("cvt.pack.sat.u16.s32 %0, %1, %2;" : "=r"(d) : "r"(hi), "r"(lo));
    return __vminu2(d, 0x01FF01FFu);
}

// Layout constants of a tile for luma sampling RH x RV (chroma 1x1):
//   4:4:4 <1,1>  MCU 8x8,   3 blocks   | 4:2:0 <2,2>  MCU 16x16, 6 blocks
//   4:2:2 <2,1>  MCU 16x8,  4 blocks   | 4:4:0 <1,2>  MCU 8x16,  4 blocks
template <int RH, int RV>
struct TileGeom
{
    static constexpr uint32_t ny = RH * RV, tot = RH * RV + 2, yh = RH;
    static constexpr uint32_t mcu_w = 8 * RH, mcu_h = 8 * RV;
    static constexpr uint32_t mcus = kTileBlocks / tot;   // MCUs per tile
    static constexpr uint32_t xg = mcu_w / 4;             // 4-pixel groups per MCU row
    static constexpr uint32_t cols = mcus * xg;           // 4-pixel columns per tile: 128, 128, 192, 96
};

constexpr uint32_t kQtStride = 68;       // words between the per-component quantiser tables: 64 + 4, so that
                                         // the three tables start in different 16-byte bank groups

// What the transform and the colour phase need to know about a tile, staged in shared memory while the
// tile's coefficients arrive.
struct TileSide
{
    alignas(16) uint32_t qt[3 * kQtStride];   // quantisers, natural order, widened to 32 bit
    uint2 mcu_xy[kTileBlocks];                // MCU coordinates inside the image (up to 192 one-block MCUs of a gray image)
    uint8_t *pix;                             // first byte of the image in the pixel plane
    uint32_t width, height;
    uint32_t mode, n_mcus;
    uint32_t samp;                            // kModeGeneric: sampling factors, one nibble each: yh | yv<<4 | uh<<8 | uv<<12 | vh<<16 | vv<<20
};

struct TileSmem
{
    // coefficient tile: kTileBlocks rows of 128 B each; the 16-byte chunk c of row r sits at chunk
    // c ^ (r & 7) (the TMA SWIZZLE_128B pattern)
    alignas(1024) uint8_t tile[kTileBlocks * 128];
    TileSide side;
    alignas(8) uint64_t bar;
};

// Chroma offsets of one pixel pair, packed as two int16: the pair shares one sample when RH == 2.
// Samples in the tile are biased by +256 (0..511), see csc_*_off_b in b2j_math.h.
template <int RH>
__device__ __forceinline__ void chroma_offsets(uint32_t cb, uint32_t cr, uint32_t &ro, uint32_t &go, uint32_t &bo, bool &special)
{
    const int32_t u0 = (int32_t)(cb & 0xFFFFu), v0 = (int32_t)(cr & 0xFFFFu);
    if (RH == 2)
    {
        ro = __byte_perm((uint32_t)csc_r_off_b(v0), 0, 0x1010);
        go = __byte_perm((uint32_t)csc_g_off_b(u0, v0), 0, 0x1010);
        bo = __byte_perm((uint32_t)csc_b_off_b(u0), 0, 0x1010);
        special = ((cb & 0xFFFFu) == 56u) & ((cr & 0xFFFFu) == 456u);   // U = -200, V = 200
    }
    else
    {
        const int32_t u1 = (int32_t)(cb >> 16), v1 = (int32_t)(cr >> 16);
        ro = __byte_perm((uint32_t)csc_r_off_b(v0), (uint32_t)csc_r_off_b(v1), 0x5410);
        go = __byte_perm((uint32_t)csc_g_off_b(u0, v0), (uint32_t)csc_g_off_b(u1, v1), 0x5410);
        bo = __byte_perm((uint32_t)csc_b_off_b(u0), (uint32_t)csc_b_off_b(u1), 0x5410);
        special = (((cb & 0xFFFFu) == 56u) & ((cr & 0xFFFFu) == 456u)) | (((cb >> 16) == 56u) & ((cr >> 16) == 456u));
    }
}

// The one double-rounding case of the reference (b2j_math.h): recompute G of a pixel pair the slow way.
__device__ __noinline__ uint32_t green_special(uint32_t yy, uint32_t cb, uint32_t cr)
{
    const int32_t ya = (int32_t)(yy & 0xFFFFu), yb = (int32_t)(yy >> 16);
    const int32_t u0 = (int32_t)(cb & 0xFFFFu), u1 = (int32_t)(cb >> 16);
    const int32_t v0 = (int32_t)(cr & 0xFFFFu), v1 = (int32_t)(cr >> 16);
    const uint32_t ga = clamp255(ya + csc_g_off_b(u0, v0) - csc_g_fix_b(ya, u0, v0));
    const uint32_t gb = clamp255(yb + csc_g_off_b(u1, v1) - csc_g_fix_b(yb, u1, v1));
    return ga | (gb << 16);
}

// Four pixels (two packed pairs per channel: value | value << 16) -> memory at d, in the output format FMT.
template <int FMT>
__device__ __forceinline__ void store_pixels4(uint8_t *__restrict__ d, size_t plane, uint32_t px, uint32_t width, bool vec_ok,
                                              const uint32_t R[2], const uint32_t Gc[2], const uint32_t B[2])
{
    if (FMT == B2J_OUT_BGRA)
    {
        uint32_t out[4];
#pragma unroll
        for (int h = 0; h < 2; h++)
        {
            const uint32_t bg = __byte_perm(B[h], Gc[h], 0x6240);     // B0 G0 B1 G1
            out[2 * h + 0] = __byte_perm(bg, R[h], 0x5410);           // B0 G0 R0 0
            out[2 * h + 1] = __byte_perm(bg, R[h], 0x7632);           // B1 G1 R1 0
        }
        if (vec_ok)
            *reinterpret_cast<uint4 *>(d) = make_uint4(out[0], out[1], out[2], out[3]);
        else
        {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (px + k < width) reinterpret_cast<uint32_t *>(d)[k] = out[k];
        }
    }
    else if (FMT == B2J_OUT_RGB24)
    {
        const uint32_t t0 = __byte_perm(R[0], Gc[0], 0x6240);         // R0 G0 R1 G1
        const uint32_t t1 = __byte_perm(R[1], Gc[1], 0x6240);         // R2 G2 R3 G3
        const uint32_t w0 = __byte_perm(t0, B[0], 0x2410);            // R0 G0 B0 R1
        const uint32_t u = __byte_perm(t0, B[0], 0x0063);             // G1 B1 . .
        const uint32_t w1 = __byte_perm(u, t1, 0x5410);               // G1 B1 R2 G2
        const uint32_t w2 = __byte_perm(t1, B[1], 0x6324);            // B2 R3 G3 B3
        if (vec_ok)
        {
            uint32_t *dw = reinterpret_cast<uint32_t *>(d);
            dw[0] = w0; dw[1] = w1; dw[2] = w2;
        }
        else
        {
            const uint32_t w[3] = {w0, w1, w2};
#pragma unroll
            for (int k = 0; k < 12; k++)
                if (px + k / 3 < width) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        }
    }
    else
    {
        const uint32_t pr = __byte_perm(R[0], R[1], 0x6420), pg = __byte_perm(Gc[0], Gc[1], 0x6420), pb = __byte_perm(B[0], B[1], 0x6420);
        if (vec_ok)
        {
            *reinterpret_cast<uint32_t *>(d) = pr;
            *reinterpret_cast<uint32_t *>(d + plane) = pg;
            *reinterpret_cast<uint32_t *>(d + 2 * plane) = pb;
        }
        else
        {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (px + k < width)
                {
                    d[k] = (uint8_t)(pr >> (8 * k)); d[plane + k] = (uint8_t)(pg >> (8 * k)); d[2 * plane + k] = (uint8_t)(pb >> (8 * k));
                }
        }
    }
}

// Colour work of one 4-pixel column of the tile for row groups [rg0, rg1) (every layout has 8 row
// groups per MCU: mcu_h / RV == 8); a work item is 4 pixels x RV rows (one chroma row). Consecutive
// threads are consecutive along x, so every store instruction writes 512 contiguous bytes per warp.
// FMT: B2J_OUT_BGRA (the reference's 32-bit pixels), B2J_OUT_RGB24 (R,G,B bytes interleaved, pitch 3W: three 32-bit
// stores per thread, 384 contiguous bytes per warp) or B2J_OUT_RGB_PLANAR (three W x H planes: one 32-bit store per plane).
template <int RH, int RV, int FMT>
__device__ __forceinline__ void csc_column(const uint8_t *__restrict__ s_tile, const TileSide &sd, uint32_t col, uint32_t rg0, uint32_t rg1)
{
    using G = TileGeom<RH, RV>;
    if (col >= sd.n_mcus * G::xg) return;
    const uint32_t width = sd.width, height = sd.height;
    const uint32_t m = col / G::xg, x4 = col % G::xg;
    const uint2 mxy = sd.mcu_xy[m];
    const uint32_t xin = x4 * 4u;
    const uint32_t px = mxy.x * G::mcu_w + xin;
    const uint32_t py_top = mxy.y * G::mcu_h;
    if (px >= width) return;
    const bool vec_ok = (width & 3u) == 0u;   // then the 4-pixel group is whole and aligned (16 / 12 / 4 bytes)
    constexpr uint32_t bpp = FMT == B2J_OUT_BGRA ? 4u : (FMT == B2J_OUT_RGB24 ? 3u : 1u);   // bytes per pixel in one plane
    const size_t pitch = (size_t)width * bpp;
    const size_t plane = (size_t)width * height;   // planar: distance between the R, G and B planes
    uint8_t *dst = sd.pix + ((size_t)py_top * width + px) * bpp;
    const uint32_t row0 = m * G::tot;
    // shared-memory addresses: luma block column and chroma blocks of this thread never change
    const uint32_t ycol = (xin >> 3), yoff = (xin & 7u) * 2u;
    const uint32_t brow = row0 + G::ny, rrow = brow + 1u;
    const uint32_t cxo = (xin / RH) * 2u;
    const uint8_t *cbp = s_tile + brow * 128u + cxo, *crp = s_tile + rrow * 128u + cxo;
    const uint32_t bsw = brow & 7u, rsw = rrow & 7u;
#pragma unroll 1
    for (uint32_t rg = rg0; rg < rg1; rg++)
    {
        if (py_top + rg * RV >= height) break;
        // chroma (pixel replication, decoder.cpp:478-480): row rg of the Cb / Cr block
        uint32_t cb2[2], cr2[2];
        if (RH == 2)
        {
            const uint32_t b = *reinterpret_cast<const uint32_t *>(cbp + ((rg ^ bsw) << 4));
            const uint32_t r = *reinterpret_cast<const uint32_t *>(crp + ((rg ^ rsw) << 4));
            cb2[0] = b & 0xFFFFu; cb2[1] = b >> 16; cr2[0] = r & 0xFFFFu; cr2[1] = r >> 16;
        }
        else
        {
            const uint2 b = *reinterpret_cast<const uint2 *>(cbp + ((rg ^ bsw) << 4));
            const uint2 r = *reinterpret_cast<const uint2 *>(crp + ((rg ^ rsw) << 4));
            cb2[0] = b.x; cb2[1] = b.y; cr2[0] = r.x; cr2[1] = r.y;
        }
        uint32_t ro[2], go[2], bo[2];
        bool sp[2];
        chroma_offsets<RH>(cb2[0], cr2[0], ro[0], go[0], bo[0], sp[0]);
        chroma_offsets<RH>(cb2[1], cr2[1], ro[1], go[1], bo[1], sp[1]);
#pragma unroll
        for (int r = 0; r < RV; r++)
        {
            const uint32_t yin = rg * RV + (uint32_t)r;
            if (r > 0 && py_top + yin >= height) break;
            const uint32_t srow = row0 + (yin >> 3) * G::yh + ycol;
            const uint2 yv = *reinterpret_cast<const uint2 *>(s_tile + srow * 128u + (((yin & 7u) ^ (srow & 7u)) << 4) + yoff);
            const uint32_t y2[2] = {yv.x, yv.y};
            uint32_t R[2], Gc[2], B[2];   // two pixels each: value | value << 16
#pragma unroll
            for (int h = 0; h < 2; h++)
            {
                R[h] = addclamp2(y2[h], ro[h]); B[h] = addclamp2(y2[h], bo[h]);
                Gc[h] = addclamp2(y2[h], go[h]);
                if (__builtin_expect(sp[h], 0))
                    Gc[h] = green_special(y2[h], RH == 2 ? cb2[h] * 0x10001u : cb2[h], RH == 2 ? cr2[h] * 0x10001u : cr2[h]);
            }
            store_pixels4<FMT>(dst + (size_t)yin * pitch, plane, px, width, vec_ok, R, Gc, B);
        }
    }
}

// Colour phase: the tile's (columns x 8 row groups) work items spread evenly over all 192 threads.
template <int RH, int RV, int FMT>
__device__ __forceinline__ void csc_phase(const uint8_t *__restrict__ s_tile, const TileSide &sd, uint32_t tid)
{
    using G = TileGeom<RH, RV>;
    if (G::cols == 192) csc_column<RH, RV, FMT>(s_tile, sd, tid, 0, 8);                                  // 4:2:2: 8 items each
    else if (G::cols == 96) csc_column<RH, RV, FMT>(s_tile, sd, tid % 96u, (tid / 96u) * 4u, (tid / 96u) * 4u + 4u);   // 4:4:0: 4 each
    else if (tid < 128) csc_column<RH, RV, FMT>(s_tile, sd, tid, 0, 5);                                  // 128 columns: 5 items ...
    else
    {
        csc_column<RH, RV, FMT>(s_tile, sd, tid - 128u, 5, 8);                                           // ... or 2 x 3 items
        csc_column<RH, RV, FMT>(s_tile, sd, tid - 64u, 5, 8);
    }
}

// Dynamic shared memory, with room to align the tile to the 1024 bytes SWIZZLE_128B needs. It stays within the 48 KB a
// kernel may use without raising cudaFuncAttributeMaxDynamicSharedMemorySize.
constexpr size_t kTileSmemBytes = sizeof(TileSmem) + 1024;
static_assert(kTileSmemBytes <= 48 * 1024, "k_idct_csc would need its dynamic shared memory limit raised");
__device__ __forceinline__ TileSmem *tile_smem()
{
    extern __shared__ uint8_t dyn_smem[];
    const uint32_t a = smem_addr(dyn_smem);
    return reinterpret_cast<TileSmem *>(dyn_smem + ((1024u - (a & 1023u)) & 1023u));
}

// Dequantise + IDCT of one block per thread, in place in the swizzled tile (decoder.cpp:340,
// cpuIDCT8x8.cpp:25-127).
// signed 16-bit x unsigned 8-bit dot product of two lanes: a.lo*b.b0 + a.hi*b.b1 (+0) and a.lo*b.b2 + a.hi*b.b3
__device__ __forceinline__ int32_t dp2a_lo(uint32_t a, uint32_t b)
{
    int32_t d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0));
    return d;
}
__device__ __forceinline__ int32_t dp2a_hi(uint32_t a, uint32_t b)
{
    int32_t d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0));
    return d;
}

// NARROWQ (every quantiser of the batch < 256, i.e. all 8-bit DQTs): the table holds one word per
// coefficient pair, q_even | q_odd << 24, and one dp2a per coefficient unpacks the int16 AND multiplies:
// dp2a.lo = c_even*q_even + c_odd*0, dp2a.hi = c_even*0 + c_odd*q_odd. Otherwise 32-bit quantisers and a
// separate unpack + multiply.
template <int RH, int RV, bool NARROWQ>
__device__ __forceinline__ void idct_phase(uint8_t *__restrict__ tilep, const TileSide &sd)
{
    using G = TileGeom<(RH > 0 ? RH : 1), (RV > 0 ? RV : 1)>;
    const uint32_t tid = threadIdx.x;
    uint32_t comp;
    if (RH == 0) comp = 0u;                   // one-component image
    else if (RH < 0)
    {
        // any other layout (kModeGeneric): block counts of the components from the sampling factors
        const uint32_t sp = sd.samp;
        const uint32_t ny = (sp & 15u) * ((sp >> 4) & 15u), nu = ((sp >> 8) & 15u) * ((sp >> 12) & 15u), nv = ((sp >> 16) & 15u) * ((sp >> 20) & 15u);
        const uint32_t bi = tid % (ny + nu + nv);
        comp = (bi >= ny ? 1u : 0u) + (bi >= ny + nu ? 1u : 0u);
    }
    else
    {
        const uint32_t bi = tid % G::tot;
        comp = bi < G::ny ? 0u : (bi - G::ny + 1u);
    }
    const uint32_t *q = sd.qt + comp * kQtStride;
    uint8_t *rowp = tilep + tid * 128u;
    const uint32_t sw = tid & 7u;
    int32_t v[64];
#pragma unroll
    for (int r = 0; r < 8; r++)
    {
        const uint4 cw = *reinterpret_cast<const uint4 *>(rowp + ((r ^ sw) << 4));
        // decoder.cpp:340: int32 product of the decoded value and the quantiser
        if (NARROWQ)
        {
            const uint4 qp = *reinterpret_cast<const uint4 *>(q + 4 * r);
            v[8 * r + 0] = dp2a_lo(cw.x, qp.x); v[8 * r + 1] = dp2a_hi(cw.x, qp.x);
            v[8 * r + 2] = dp2a_lo(cw.y, qp.y); v[8 * r + 3] = dp2a_hi(cw.y, qp.y);
            v[8 * r + 4] = dp2a_lo(cw.z, qp.z); v[8 * r + 5] = dp2a_hi(cw.z, qp.z);
            v[8 * r + 6] = dp2a_lo(cw.w, qp.w); v[8 * r + 7] = dp2a_hi(cw.w, qp.w);
        }
        else
        {
            const uint4 qa = *reinterpret_cast<const uint4 *>(q + 8 * r);
            const uint4 qb = *reinterpret_cast<const uint4 *>(q + 8 * r + 4);
            v[8 * r + 0] = (int32_t)(int16_t)(cw.x & 0xFFFFu) * (int32_t)qa.x;
            v[8 * r + 1] = ((int32_t)cw.x >> 16) * (int32_t)qa.y;
            v[8 * r + 2] = (int32_t)(int16_t)(cw.y & 0xFFFFu) * (int32_t)qa.z;
            v[8 * r + 3] = ((int32_t)cw.y >> 16) * (int32_t)qa.w;
            v[8 * r + 4] = (int32_t)(int16_t)(cw.z & 0xFFFFu) * (int32_t)qb.x;
            v[8 * r + 5] = ((int32_t)cw.z >> 16) * (int32_t)qb.y;
            v[8 * r + 6] = (int32_t)(int16_t)(cw.w & 0xFFFFu) * (int32_t)qb.z;
            v[8 * r + 7] = ((int32_t)cw.w >> 16) * (int32_t)qb.w;
        }
        idct_row(v[8 * r + 0], v[8 * r + 1], v[8 * r + 2], v[8 * r + 3], v[8 * r + 4], v[8 * r + 5], v[8 * r + 6], v[8 * r + 7]);
    }
    // the +256 sample bias enters through the DC row: the column pass computes (b0*256 + 8192 + ...) >> 14, and
    // 256 << 14 == 16384 * 256, so adding 16384 to b0 adds exactly 256 to all eight outputs of the column
#pragma unroll
    for (int c = 0; c < 8; c++)
    {
        v[c] += 16384;
        idct_col_noclip(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c]);
    }
#pragma unroll
    for (int r = 0; r < 8; r++)
    {
        uint4 o;
        o.x = pack_clip2(v[8 * r + 0], v[8 * r + 1]);
        o.y = pack_clip2(v[8 * r + 2], v[8 * r + 3]);
        o.z = pack_clip2(v[8 * r + 4], v[8 * r + 5]);
        o.w = pack_clip2(v[8 * r + 6], v[8 * r + 7]);
        *reinterpret_cast<uint4 *>(rowp + ((r ^ sw) << 4)) = o;
    }
}

template <bool NARROWQ>
__device__ __forceinline__ void idct_dispatch(uint8_t *tilep, const TileSide &sd)
{
    switch (sd.mode)   // uniform per CTA
    {
    case kMode444: idct_phase<1, 1, NARROWQ>(tilep, sd); break;
    case kMode420: idct_phase<2, 2, NARROWQ>(tilep, sd); break;
    case kMode422: idct_phase<2, 1, NARROWQ>(tilep, sd); break;
    default:       idct_phase<1, 2, NARROWQ>(tilep, sd); break;
    }
}

// chroma replication + colour + store (decoder.cpp:443-495, 367-370)
// One-component images (kModeGray): a tile is 192 one-block MCUs; an item is 4 pixels x 8 rows of one block.
// YUV_to_RGB32 with U = V = 0 (decoder.cpp:367-370): R = G = B = clamp(Y + 128).
template <int FMT>
__device__ __forceinline__ void csc_gray(const uint8_t *__restrict__ s_tile, const TileSide &sd, uint32_t tid)
{
    const uint32_t width = sd.width, height = sd.height;
    const bool vec_ok = (width & 3u) == 0u;
    constexpr uint32_t bpp = FMT == B2J_OUT_BGRA ? 4u : (FMT == B2J_OUT_RGB24 ? 3u : 1u);
    const size_t pitch = (size_t)width * bpp, plane = (size_t)width * height;
    for (uint32_t it = tid; it < sd.n_mcus * 2u; it += kTileBlocks)
    {
        const uint32_t m = it >> 1, xin = (it & 1u) * 4u;
        const uint2 mxy = sd.mcu_xy[m];
        const uint32_t px = mxy.x * 8u + xin, py = mxy.y * 8u;
        if (px >= width) continue;
        uint8_t *dst = sd.pix + ((size_t)py * width + px) * bpp;
#pragma unroll 1
        for (uint32_t r = 0; r < 8u && py + r < height; r++)
        {
            const uint2 yv = *reinterpret_cast<const uint2 *>(s_tile + m * 128u + ((r ^ (m & 7u)) << 4) + xin * 2u);
            // samples carry the +256 bias of the IDCT phase: Y + 128 = Yb - 128
            const uint32_t g[2] = {addclamp2(yv.x, 0xFF80FF80u), addclamp2(yv.y, 0xFF80FF80u)};
            store_pixels4<FMT>(dst + (size_t)r * pitch, plane, px, width, vec_ok, g, g, g);
        }
    }
}

// Any other layout (kModeGeneric; SURVEY.md 8f rank 4): luma h x v with chroma components whose factors divide the
// luma's -- 4:1:1 (41,11,11), 14, 31, 42, ..., and components with several blocks per MCU (22,21,21). The reference's
// generic loop (decoder.cpp:474-483), one 4-pixel group per work item, one pixel at a time: rare layouts, kept simple.
template <int FMT>
__device__ __forceinline__ void csc_generic(const uint8_t *__restrict__ s_tile, const TileSide &sd, uint32_t tid)
{
    const uint32_t sp = sd.samp;
    const uint32_t yh = sp & 15u, yv = (sp >> 4) & 15u, uh = (sp >> 8) & 15u, uv = (sp >> 12) & 15u, vh = (sp >> 16) & 15u, vv = (sp >> 20) & 15u;
    const uint32_t ny = yh * yv, nu = uh * uv, tot = ny + nu + vh * vv;
    const uint32_t mcu_w = 8u * yh, mcu_h = 8u * yv, xg = mcu_w / 4u, items = mcu_h * xg;
    const uint32_t ruh = yh / uh, ruv = yv / uv, rvh = yh / vh, rvv = yv / vv;
    const uint32_t width = sd.width, height = sd.height;
    const bool vec_ok = (width & 3u) == 0u;
    constexpr uint32_t bpp = FMT == B2J_OUT_BGRA ? 4u : (FMT == B2J_OUT_RGB24 ? 3u : 1u);
    const size_t plane = (size_t)width * height;
    for (uint32_t it = tid; it < sd.n_mcus * items; it += kTileBlocks)
    {
        const uint32_t m = it / items, r = it % items, y = r / xg, x = (r % xg) * 4u;
        const uint2 mxy = sd.mcu_xy[m];
        const uint32_t px = mxy.x * mcu_w + x, py = mxy.y * mcu_h + y;
        if (px >= width || py >= height) continue;
        const uint32_t row0 = m * tot;
        uint32_t rgb[4];
#pragma unroll
        for (uint32_t k = 0; k < 4u; k++)
        {
            const uint32_t xx = x + k;
            const uint32_t yb = row0 + (y >> 3) * yh + (xx >> 3);
            const uint32_t ux = xx / ruh, uy = y / ruv, vx = xx / rvh, vy = y / rvv;
            const uint32_t ub = row0 + ny + (uy >> 3) * uh + (ux >> 3), vb = row0 + ny + nu + (vy >> 3) * vh + (vx >> 3);
            const uint32_t Y = *reinterpret_cast<const uint16_t *>(s_tile + yb * 128u + (((y & 7u) ^ (yb & 7u)) << 4) + (xx & 7u) * 2u);
            const uint32_t U = *reinterpret_cast<const uint16_t *>(s_tile + ub * 128u + (((uy & 7u) ^ (ub & 7u)) << 4) + (ux & 7u) * 2u);
            const uint32_t V = *reinterpret_cast<const uint16_t *>(s_tile + vb * 128u + (((vy & 7u) ^ (vb & 7u)) << 4) + (vx & 7u) * 2u);
            rgb[k] = csc_pixel_biased((int32_t)Y, (int32_t)U, (int32_t)V);   // R << 16 | G << 8 | B
        }
        uint32_t R[2], Gc[2], B[2];
#pragma unroll
        for (int h = 0; h < 2; h++)
        {
            R[h] = (rgb[2 * h] >> 16) | (rgb[2 * h + 1] >> 16) << 16;
            Gc[h] = ((rgb[2 * h] >> 8) & 0xFFu) | ((rgb[2 * h + 1] >> 8) & 0xFFu) << 16;
            B[h] = (rgb[2 * h] & 0xFFu) | (rgb[2 * h + 1] & 0xFFu) << 16;
        }
        store_pixels4<FMT>(sd.pix + ((size_t)py * width + px) * bpp, plane, px, width, vec_ok, R, Gc, B);
    }
}

template <int FMT>
__device__ __forceinline__ void csc_dispatch(const uint8_t *tilep, const TileSide &sd)
{
    const uint32_t tid = threadIdx.x;
    switch (sd.mode)
    {
    case kMode444: csc_phase<1, 1, FMT>(tilep, sd, tid); break;
    case kMode420: csc_phase<2, 2, FMT>(tilep, sd, tid); break;
    case kMode422: csc_phase<2, 1, FMT>(tilep, sd, tid); break;
    default:       csc_phase<1, 2, FMT>(tilep, sd, tid); break;
    }
}

// Side data of a tile: every global load first, then the stores to shared memory.
template <bool NARROWQ>
__device__ __forceinline__ void side_stage(TileSide &sd, const ImgDev *__restrict__ imgs, const uint16_t *__restrict__ qtabs, const TileDev d,
                                           uint8_t *__restrict__ pix)
{
    const uint32_t tid = threadIdx.x;
    const ImgDev *im = imgs + d.img;
    const uint32_t q = tid < 96 ? __ldg(reinterpret_cast<const uint32_t *>(qtabs + (size_t)d.img * 192) + tid) : 0u;   // a pair
    const uint32_t width = __ldg(&im->width);
    const uint32_t height = __ldg(&im->height);
    const uint32_t mcu_count_w = __ldg(&im->mcu_count_w);
    const uint32_t samp = __ldg(&im->samp);
    const uint64_t pix_off = __ldg(reinterpret_cast<const unsigned long long *>(&im->pix_off));
    const uint32_t n_mcus = d.info >> 8;
    if (tid < 96)
    {
        const uint32_t comp = tid >> 5, k = tid & 31u;   // quantiser pair k of component comp
        if (NARROWQ) sd.qt[comp * kQtStride + k] = (q & 0xFFu) | ((q >> 16) << 24);
        else { sd.qt[comp * kQtStride + 2 * k] = q & 0xFFFFu; sd.qt[comp * kQtStride + 2 * k + 1] = q >> 16; }
    }
    if (tid < n_mcus)
    {
        const uint32_t gm = d.mcu_first + tid;
        const uint32_t my = gm / mcu_count_w;
        sd.mcu_xy[tid] = make_uint2(gm - my * mcu_count_w, my);
    }
    if (tid == 0)
    {
        sd.pix = pix + pix_off;
        sd.width = width; sd.height = height;
        sd.mode = d.info & 0xFFu; sd.n_mcus = n_mcus;
        sd.samp = samp;
    }
}

// The CTA's tile (tiles[blockIdx.x], returned): its 24 KB of coefficients arrive in sm.tile by one TMA tensor load
// (128-byte swizzle, mbarrier completion) issued by thread 0 while the other threads stage the side data. The wait is
// bounded: a load that never completes flags the image with B2J_ST_INTERNAL.
template <bool NARROWQ>
__device__ __forceinline__ TileDev tile_load(TileSmem &sm, const CUtensorMap *tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
                                             const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ pix, int32_t *__restrict__ status)
{
    const uint32_t tid = threadIdx.x;
    const TileDev d = tiles[blockIdx.x];
    if (tid == 0)
    {
        mbar_init(&sm.bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(&sm.bar, kTileBlocks * 128);
        tma_load_2d(sm.tile, tmap, 0, (int)d.row_first, &sm.bar);
    }
    side_stage<NARROWQ>(sm.side, imgs, qtabs, d, pix);
    __syncthreads();   // barrier initialisation + side data visible
    uint32_t spins = 0;
    while (!mbar_try_wait(&sm.bar, 0))
    {
        if (++spins > (1u << 22)) { if (tid == 0) atomicOr(&status[d.img], B2J_ST_INTERNAL); break; }   // never hang the GPU
    }
    return d;
}

// One tile per CTA, loaded by tile_load.
// Measured on B200 (profiles/): a persistent double-buffered variant and a warp-autonomous variant of
// this kernel were both slower -- the kernel is bound by dependent-issue latency at 24 warps per SM,
// not by the latency in front of a tile, so the simplest structure wins.
constexpr int kIdctMinCtas = 5;   // measured on B200: 64 registers with ~220 B of spills beats 80 registers at 4 CTAs per SM
// KIND: kTileColour (the four everyday layouts), kTileGray (one-component images, B2J_GATE_GRAY) or kTileGeneric (any
// other layout: csc_generic). Each kind is a kernel of its own over a tile range of its own (the host sorts the batch's
// tiles by kind), because merely carrying the extra paths, or a test for them at the top of the kernel, slows the
// colour kernel down by 2 % (measured).
constexpr int kTileColour = 0, kTileGray = 1, kTileGeneric = 2;
template <bool NARROWQ, int FMT, int KIND>
__global__ void __launch_bounds__(kTileBlocks, kIdctMinCtas)
k_idct_csc(const __grid_constant__ CUtensorMap tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
           const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ pix, int32_t *__restrict__ status)
{
    TileSmem &sm = *tile_smem();
    const uint32_t tid = threadIdx.x;
    tile_load<NARROWQ>(sm, &tmap, imgs, tiles, qtabs, pix, status);
    if (KIND == kTileGray)
    {
        idct_phase<0, 0, NARROWQ>(sm.tile, sm.side);
        __syncthreads();
        csc_gray<FMT>(sm.tile, sm.side, tid);
    }
    else if (KIND == kTileGeneric)
    {
        idct_phase<-1, -1, NARROWQ>(sm.tile, sm.side);
        __syncthreads();
        csc_generic<FMT>(sm.tile, sm.side, tid);
    }
    else
    {
        idct_dispatch<NARROWQ>(sm.tile, sm.side);
        __syncthreads();
        csc_dispatch<FMT>(sm.tile, sm.side);
    }
}

// =====================================================================================
// The libjpeg pixel model (B2J_PIXELS_LIBJPEG): libjpeg-turbo's default decode of the same coefficients at scale_denom
// s = 1, 2, 4 or 8 (b2j_batch_set_scale), in two kernels of their own so that the reference model's colour kernel keeps
// its code and its instruction cache (DESIGN.md §3). Both take the smallest DCT size MINS = 8 / s as a template parameter.
//   k_idct_libjpeg      per tile, one thread per block: dequantise, then at the component's DCT size ss (jdmaster.c)
//                       the ISLOW IDCT (jidctint.c, ss 8) or a reduced one (jidctred.c), range limit; ss x ss samples
//                       per block into the sample plane
//   k_upsample_libjpeg  per 4-pixel group of the ceil(W / s) x ceil(H / s) output: chroma upsampling as jdsample.c
//                       chooses it (fancy triangle filter for 2x1, 2x2 and 1x2 while MINS > 1, replication otherwise),
//                       fixed-point YCbCr -> RGB (jdcolor.c), store in the output format
// Sample plane: image i at byte 64 * blk_first, its components one after another, each with a share of 64 bytes per
// block, so the image's share is 64 * blk_count. A component of DCT size ss fills (mcu_count_w * h * ss) x
// (mcu_count_h * v * ss) bytes at the start of its share: at ss 8, all of it.

// One 1-D pass of jpeg_idct_islow (CONST_BITS 13) over d[0..7] (a column, then a row), in place, descaled by N bits.
// The arithmetic is 64-bit, like libjpeg's JLONG: a dequantised coefficient reaches 32767 * 65535 < 2^31, and the
// constants reach 2^14.7, so 32-bit products would overflow for the large coefficients valid files may carry.
template <int N>
__device__ __forceinline__ void islow_1d(int64_t d[8])
{
    int64_t z1 = (d[2] + d[6]) * 4433;                      // FIX(0.541196100)
    const int64_t tmp2 = z1 - d[6] * 15137;                 // FIX(1.847759065)
    const int64_t tmp3 = z1 + d[2] * 6270;                  // FIX(0.765366865)
    const int64_t tmp0 = (d[0] + d[4]) * 8192, tmp1 = (d[0] - d[4]) * 8192;
    const int64_t e10 = tmp0 + tmp3, e13 = tmp0 - tmp3, e11 = tmp1 + tmp2, e12 = tmp1 - tmp2;
    int64_t t0 = d[7], t1 = d[5], t2 = d[3], t3 = d[1];
    z1 = t0 + t3;
    int64_t z2 = t1 + t2, z3 = t0 + t2, z4 = t1 + t3;
    const int64_t z5 = (z3 + z4) * 9633;                    // FIX(1.175875602)
    t0 *= 2446; t1 *= 16819; t2 *= 25172; t3 *= 12299;      // FIX(0.298631336), FIX(2.053119869), FIX(3.072711026), FIX(1.501321110)
    z1 *= -7373; z2 *= -20995;                              // FIX(0.899976223), FIX(2.562915447)
    z3 = z3 * -16069 + z5; z4 = z4 * -3196 + z5;            // FIX(1.961570560), FIX(0.390180644)
    t0 += z1 + z3; t1 += z2 + z4; t2 += z2 + z3; t3 += z1 + z4;
    constexpr int64_t r = 1ll << (N - 1);
    d[0] = (e10 + t3 + r) >> N; d[7] = (e10 - t3 + r) >> N;
    d[1] = (e11 + t2 + r) >> N; d[6] = (e11 - t2 + r) >> N;
    d[2] = (e12 + t1 + r) >> N; d[5] = (e12 - t1 + r) >> N;
    d[3] = (e13 + t0 + r) >> N; d[4] = (e13 - t0 + r) >> N;
}

// libjpeg's range limit of an IDCT output (sample_range_limit[] indexed with y & 1023): it wraps, it does not clamp.
__device__ __forceinline__ uint32_t islow_limit(int64_t y)
{
    const uint32_t m = ((uint32_t)y + 128u) & 1023u;
    return m < 256u ? m : (m < 640u ? 255u : 0u);
}

// Dequantised coefficient (r, c) of the block in tile row `rowp` (swizzle sw): DEQUANTIZE, an int product (fits, see islow_1d).
__device__ __forceinline__ int64_t tile_coef(const uint8_t *rowp, uint32_t sw, const uint32_t *q, int r, int c)
{
    const int32_t coef = *reinterpret_cast<const int16_t *>(rowp + (((uint32_t)r ^ sw) << 4) + c * 2);
    return (int64_t)(coef * (int32_t)q[8 * r + c]);
}

// jpeg_idct_islow of the block in row `row` of the tile: 8 rows of 8 samples at dst, `pitch` bytes apart (pitch and dst
// multiples of 8).
__device__ __forceinline__ void islow_block(const uint8_t *tile, uint32_t row, const uint32_t *q, uint8_t *dst, size_t pitch)
{
    const uint8_t *rowp = tile + row * 128u;
    const uint32_t sw = row & 7u;
    int32_t ws[64];   // jidctint.c's int workspace: the pass-1 results are stored as 32-bit ints
#pragma unroll
    for (int c = 0; c < 8; c++)
    {
        int64_t col[8];
#pragma unroll
        for (int r = 0; r < 8; r++) col[r] = tile_coef(rowp, sw, q, r, c);
        islow_1d<13 - 2>(col);
#pragma unroll
        for (int r = 0; r < 8; r++) ws[8 * r + c] = (int32_t)col[r];
    }
#pragma unroll
    for (int r = 0; r < 8; r++)
    {
        int64_t row8[8];
#pragma unroll
        for (int c = 0; c < 8; c++) row8[c] = ws[8 * r + c];
        islow_1d<13 + 2 + 3>(row8);
        uint2 o;
        o.x = islow_limit(row8[0]) | islow_limit(row8[1]) << 8 | islow_limit(row8[2]) << 16 | islow_limit(row8[3]) << 24;
        o.y = islow_limit(row8[4]) | islow_limit(row8[5]) << 8 | islow_limit(row8[6]) << 16 | islow_limit(row8[7]) << 24;
        *reinterpret_cast<uint2 *>(dst + (size_t)r * pitch) = o;
    }
}

// A component's DCT size ss as jdmaster.c chooses it for the smallest size mins = 8 / scale: doubled from mins while
// both of its factors still divide the maxima evenly. Its blocks become ss x ss samples; 4:2:0 at 1/2: luma 4, chroma 8.
__device__ __forceinline__ uint32_t dct_size(uint32_t h, uint32_t v, uint32_t hmax, uint32_t vmax, uint32_t mins)
{
    uint32_t ss = mins;
    while (ss < 8u && (hmax * mins) % (h * ss * 2u) == 0u && (vmax * mins) % (v * ss * 2u) == 0u) ss *= 2u;
    return ss;
}

// One 1-D pass of jidctred.c's jpeg_idct_4x4 over d[0..7] (d[4] is not used): 4 outputs, descaled by N bits.
template <int N>
__device__ __forceinline__ void red4_1d(const int64_t d[8], int64_t o[4])
{
    const int64_t t0 = d[0] * (1ll << 14);                   // << (CONST_BITS + 1)
    const int64_t t2 = d[2] * 15137 - d[6] * 6270;           // FIX(1.847759065), FIX(0.765366865)
    const int64_t t10 = t0 + t2, t12 = t0 - t2;
    const int64_t a = d[7] * -1730 + d[5] * 11893 + d[3] * -17799 + d[1] * 8697;   // FIX(0.211164243), FIX(1.451774981), FIX(2.172734803), FIX(1.061594337)
    const int64_t b = d[7] * -4176 + d[5] * -4926 + d[3] * 7373 + d[1] * 20995;    // FIX(0.509795579), FIX(0.601344887), FIX(0.899976223), FIX(2.562915447)
    constexpr int64_t r = 1ll << (N - 1);
    o[0] = (t10 + b + r) >> N; o[3] = (t10 - b + r) >> N;
    o[1] = (t12 + a + r) >> N; o[2] = (t12 - a + r) >> N;
}

// One 1-D pass of jpeg_idct_2x2 over d[0], d[1], d[3], d[5], d[7]: 2 outputs, descaled by N bits.
template <int N>
__device__ __forceinline__ void red2_1d(const int64_t d[8], int64_t o[2])
{
    const int64_t t10 = d[0] * (1ll << 15);                  // << (CONST_BITS + 2)
    const int64_t t0 = d[7] * -5906 + d[5] * 6967 + d[3] * -10426 + d[1] * 29692;  // FIX(0.720959822), FIX(0.850430095), FIX(1.272758580), FIX(3.624509785)
    constexpr int64_t r = 1ll << (N - 1);
    o[0] = (t10 + t0 + r) >> N; o[1] = (t10 - t0 + r) >> N;
}

// jpeg_idct_4x4: 4 rows of 4 samples at dst (pitch and dst multiples of 4). Like islow_block, 64-bit products and a
// 32-bit workspace; column 4 contributes nothing.
__device__ __forceinline__ void red4_block(const uint8_t *tile, uint32_t row, const uint32_t *q, uint8_t *dst, size_t pitch)
{
    const uint8_t *rowp = tile + row * 128u;
    const uint32_t sw = row & 7u;
    int32_t ws[4][8];
#pragma unroll
    for (int c = 0; c < 8; c++)
    {
        if (c == 4) continue;
        int64_t col[8], o[4];
#pragma unroll
        for (int r = 0; r < 8; r++) col[r] = r == 4 ? 0 : tile_coef(rowp, sw, q, r, c);
        red4_1d<13 - 2 + 1>(col, o);
#pragma unroll
        for (int r = 0; r < 4; r++) ws[r][c] = (int32_t)o[r];
    }
#pragma unroll
    for (int r = 0; r < 4; r++)
    {
        int64_t d[8], o[4];
#pragma unroll
        for (int c = 0; c < 8; c++) d[c] = c == 4 ? 0 : ws[r][c];
        red4_1d<13 + 2 + 3 + 1>(d, o);
        *reinterpret_cast<uint32_t *>(dst + (size_t)r * pitch) =
            islow_limit(o[0]) | islow_limit(o[1]) << 8 | islow_limit(o[2]) << 16 | islow_limit(o[3]) << 24;
    }
}

// jpeg_idct_2x2: 2 rows of 2 samples at dst (pitch and dst even); only rows and columns 0, 1, 3, 5 and 7 contribute.
__device__ __forceinline__ void red2_block(const uint8_t *tile, uint32_t row, const uint32_t *q, uint8_t *dst, size_t pitch)
{
    const uint8_t *rowp = tile + row * 128u;
    const uint32_t sw = row & 7u;
    constexpr uint32_t kUsed = 0xABu;   // bits 0, 1, 3, 5, 7
    int32_t ws[2][8];
#pragma unroll
    for (int c = 0; c < 8; c++)
    {
        if (!((kUsed >> c) & 1u)) continue;
        int64_t col[8], o[2];
#pragma unroll
        for (int r = 0; r < 8; r++) col[r] = ((kUsed >> r) & 1u) ? tile_coef(rowp, sw, q, r, c) : 0;
        red2_1d<13 - 2 + 2>(col, o);
        ws[0][c] = (int32_t)o[0]; ws[1][c] = (int32_t)o[1];
    }
#pragma unroll
    for (int r = 0; r < 2; r++)
    {
        int64_t d[8], o[2];
#pragma unroll
        for (int c = 0; c < 8; c++) d[c] = ((kUsed >> c) & 1u) ? ws[r][c] : 0;
        red2_1d<13 + 2 + 3 + 2>(d, o);
        *reinterpret_cast<uint16_t *>(dst + (size_t)r * pitch) = (uint16_t)(islow_limit(o[0]) | islow_limit(o[1]) << 8);
    }
}

// Every tile kind in one kernel: the component of a block comes from the image's sampling factors (gray: 0x11, one
// block). Every block becomes ss x ss samples of its component's plane (pitch mcu_count_w * h * ss), by jpeg_idct_islow
// (ss 8), jidctred.c's reduced transforms or jpeg_idct_1x1: (DC * q + 4) >> 3. Threads take the tile's blocks component
// by component (the luma blocks of all its MCUs, then Cb's, then Cr's), so that a warp mixes transform sizes only where
// one component's run ends inside it: never in a full 4:2:0 tile (128 luma, 32 + 32 chroma blocks). MINS, the smallest
// DCT size, is a template parameter so that the full-size decode (MINS 8) carries no reduced transform.
template <uint32_t MINS>
__global__ void __launch_bounds__(kTileBlocks)
k_idct_libjpeg(const __grid_constant__ CUtensorMap tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
               const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ samples, int32_t *__restrict__ status)
{
    TileSmem &sm = *tile_smem();
    const uint32_t tid = threadIdx.x;
    const TileDev d = tile_load<false>(sm, &tmap, imgs, tiles, qtabs, samples, status);   // 32-bit quantisers; sd.pix is not used
    const ImgDev *im = imgs + d.img;
    const uint32_t sp = sm.side.samp, n = sm.side.n_mcus;
    const uint32_t yh = sp & 15u, yv = (sp >> 4) & 15u, uh = (sp >> 8) & 15u, uv = (sp >> 12) & 15u, vh = (sp >> 16) & 15u, vv = (sp >> 20) & 15u;
    const uint32_t ny = yh * yv, nu = uh * uv, tot = ny + nu + vh * vv;
    if (tid >= n * tot) return;
    const uint32_t comp = (tid >= n * ny ? 1u : 0u) + (tid >= n * (ny + nu) ? 1u : 0u);
    const uint32_t before = (comp > 0 ? ny : 0u) + (comp > 1 ? nu : 0u);   // blocks of the earlier components per MCU
    const uint32_t nc = comp == 0 ? ny : (comp == 1 ? nu : vh * vv);
    const uint32_t j = tid - n * before, m = j / nc, k = j % nc;        // MCU m of the tile, block k of the component in it
    const uint32_t h = comp == 0 ? yh : (comp == 1 ? uh : vh), v = comp == 0 ? yv : (comp == 1 ? uv : vv);
    const uint32_t ss = dct_size(h, v, yh, yv, MINS);   // the chroma factors divide the luma's (geometry_ok): those are the maxima
    const uint32_t mcu_count = __ldg(&im->mcu_count), mcw = __ldg(&im->mcu_count_w), blk_first = __ldg(&im->blk_first);
    const size_t pitch = (size_t)mcw * h * ss;
    const uint2 mxy = sm.side.mcu_xy[m];
    uint8_t *dst = samples + 64ull * ((size_t)blk_first + (size_t)mcu_count * before) + (size_t)((mxy.y * v + k / h) * ss) * pitch +
                   (mxy.x * h + k % h) * ss;
    const uint32_t row = m * tot + before + k;   // the block's row in the tile (MCU-interleaved)
    const uint32_t *q = sm.side.qt + comp * kQtStride;
    if (ss == 8u) islow_block(sm.tile, row, q, dst, pitch);
    else if (ss == 4u) red4_block(sm.tile, row, q, dst, pitch);
    else if (ss == 2u) red2_block(sm.tile, row, q, dst, pitch);
    else *dst = (uint8_t)islow_limit((tile_coef(sm.tile + row * 128u, row & 7u, q, 0, 0) + 4) >> 3);
}

// One component of an image in the sample plane, and how it becomes output resolution.
struct UpComp
{
    const uint8_t *p;     // first sample of the component's plane
    uint32_t pitch;       // bytes per row of the plane
    uint32_t dw, dh;      // samples that belong to the image (up_comp)
    uint32_t rh, rv;      // upsampling ratios (up_comp)
};

// A component of DCT size ss (dct_size) has ceil(W * h * ss / (hmax * 8)) x ceil(H * v * ss / (vmax * 8)) samples (jdmaster.c's
// downsampled_width / _height) and is upsampled by hmax * mins / (h * ss) x vmax * mins / (v * ss).
__device__ __forceinline__ UpComp up_comp(const uint8_t *p, uint32_t h, uint32_t v, uint32_t hmax, uint32_t vmax, uint32_t mcw,
                                          uint32_t width, uint32_t height, uint32_t mins)
{
    const uint32_t ss = dct_size(h, v, hmax, vmax, mins);
    UpComp c;
    c.p = p; c.pitch = mcw * h * ss;
    c.dw = (width * h * ss + hmax * 8u - 1u) / (hmax * 8u); c.dh = (height * v * ss + vmax * 8u - 1u) / (vmax * 8u);
    c.rh = hmax * mins / (h * ss); c.rv = vmax * mins / (v * ss);
    return c;
}

// The component's value at output pixel (x, y), as jdsample.c computes it. Neighbours outside [0, dw) x [0, dh) are
// clamped, which is libjpeg's edge replication; the first and last columns of its loops are that case. jdsample.c
// applies its fancy filters only while the smallest DCT size exceeds 1 (`fancy`): at 1/8 every ratio replicates.
__device__ __forceinline__ uint32_t up_sample(const UpComp &c, uint32_t x, uint32_t y, bool fancy)
{
    if (fancy)
    {
        const bool fancy_h = c.rh == 2u && c.dw > 2u;
        if (c.rh == 1u && c.rv == 1u) return __ldg(c.p + (size_t)y * c.pitch + x);
        if (c.rh == 1u && c.rv == 2u)                                      // h1v2_fancy_upsample
        {
            const uint32_t r = y >> 1, n = (y & 1u) ? min(r + 1u, c.dh - 1u) : (r ? r - 1u : 0u);
            return (3u * __ldg(c.p + (size_t)r * c.pitch + x) + __ldg(c.p + (size_t)n * c.pitch + x) + 1u + (y & 1u)) >> 2;
        }
        if (fancy_h && c.rv == 1u)                                         // h2v1_fancy_upsample
        {
            const uint8_t *row = c.p + (size_t)y * c.pitch;
            const uint32_t sx = x >> 1, nx = (x & 1u) ? min(sx + 1u, c.dw - 1u) : (sx ? sx - 1u : 0u);
            return (3u * __ldg(row + sx) + __ldg(row + nx) + 1u + (x & 1u)) >> 2;
        }
        if (fancy_h && c.rv == 2u)                                         // h2v2_fancy_upsample
        {
            const uint32_t r = y >> 1, n = (y & 1u) ? min(r + 1u, c.dh - 1u) : (r ? r - 1u : 0u);
            const uint32_t sx = x >> 1, nx = (x & 1u) ? min(sx + 1u, c.dw - 1u) : (sx ? sx - 1u : 0u);
            const uint8_t *r0 = c.p + (size_t)r * c.pitch, *r1 = c.p + (size_t)n * c.pitch;
            const uint32_t cs = 3u * __ldg(r0 + sx) + __ldg(r1 + sx), cn = 3u * __ldg(r0 + nx) + __ldg(r1 + nx);
            return (3u * cs + cn + 8u - (x & 1u)) >> 4;
        }
    }
    return __ldg(c.p + (size_t)(y / c.rv) * c.pitch + x / c.rh);          // int_upsample / h2v1 / h2v2: replication
}

// jdcolor.c ycc_rgb_convert (SCALEBITS 16): R | G << 8 | B << 16
__device__ __forceinline__ uint32_t ycc_rgb_libjpeg(int32_t y, int32_t cb, int32_t cr)
{
    cb -= 128; cr -= 128;
    const int32_t r = y + ((91881 * cr + 32768) >> 16);
    const int32_t g = y + ((-22554 * cb - 46802 * cr + 32768) >> 16);
    const int32_t b = y + ((116130 * cb + 32768) >> 16);
    return (uint32_t)min(max(r, 0), 255) | (uint32_t)min(max(g, 0), 255) << 8 | (uint32_t)min(max(b, 0), 255) << 16;
}

// 4-pixel group i of the width x height window at (x0, y0) of an image's ceil(W / s) x ceil(H / s) output, s = 8 / MINS,
// into the window's pixels at the image's pix_off (pitch: the window's width). The samples are read in the image's whole
// sample plane, so the fancy filters at the window's edges see the neighbours outside it, clamped at the image's edges.
template <int FMT, uint32_t MINS>
__device__ __forceinline__ void upsample_group(const uint8_t *__restrict__ samples, const ImgDev &im, uint32_t x0, uint32_t y0, uint32_t width,
                                               uint32_t height, uint32_t i, uint8_t *__restrict__ pix)
{
    constexpr bool fancy = MINS > 1u;
    const uint32_t gw = (width + 3u) / 4u;
    if (i >= gw * height) return;
    const uint32_t py = i / gw, px = (i % gw) * 4u;
    const uint32_t sp = im.samp, mcw = im.mcu_count_w;
    const uint32_t yh = sp & 15u, yv = (sp >> 4) & 15u, uh = (sp >> 8) & 15u, uv = (sp >> 12) & 15u, vh = (sp >> 16) & 15u, vv = (sp >> 20) & 15u;
    const uint8_t *p0 = samples + 64ull * im.blk_first;
    const bool gray = im.mode == kModeGray;
    // the chroma factors divide the luma's (geometry_ok), so the luma's are the maxima
    const UpComp cy = up_comp(p0, yh, yv, yh, yv, mcw, im.width, im.height, MINS);
    UpComp cu = cy, cv = cy;
    if (!gray)
    {
        cu = up_comp(p0 + 64ull * im.mcu_count * (yh * yv), uh, uv, yh, yv, mcw, im.width, im.height, MINS);
        cv = up_comp(p0 + 64ull * im.mcu_count * (yh * yv + uh * uv), vh, vv, yh, yv, mcw, im.width, im.height, MINS);
    }
    uint32_t R[2] = {0u, 0u}, Gc[2] = {0u, 0u}, B[2] = {0u, 0u};
#pragma unroll
    for (uint32_t k = 0; k < 4u; k++)
    {
        const uint32_t x = x0 + min(px + k, width - 1u), y = y0 + py;   // the stores skip pixels behind the last column
        const uint32_t Y = up_sample(cy, x, y, fancy);
        const uint32_t rgb = gray ? Y * 0x10101u
                                  : ycc_rgb_libjpeg((int32_t)Y, (int32_t)up_sample(cu, x, y, fancy), (int32_t)up_sample(cv, x, y, fancy));
        const uint32_t sh = 16u * (k & 1u);
        R[k >> 1] |= (rgb & 0xFFu) << sh; Gc[k >> 1] |= ((rgb >> 8) & 0xFFu) << sh; B[k >> 1] |= (rgb >> 16) << sh;
    }
    constexpr uint32_t bpp = FMT == B2J_OUT_BGRA ? 4u : (FMT == B2J_OUT_RGB24 ? 3u : 1u);
    store_pixels4<FMT>(pix + im.pix_off + ((size_t)py * width + px) * bpp, (size_t)width * height, px, width, (width & 3u) == 0u, R, Gc, B);
}

// One thread per 4-pixel group of a row of the ceil(W / s) x ceil(H / s) output, s = 8 / MINS; blockIdx.y (strided by
// gridDim.y) = image.
template <int FMT, uint32_t MINS>
__global__ void __launch_bounds__(256)
k_upsample_libjpeg(const uint8_t *__restrict__ samples, const ImgDev *__restrict__ imgs, uint32_t n_images, uint8_t *__restrict__ pix)
{
    constexpr uint32_t s = 8u / MINS;
    for (uint32_t img = blockIdx.y; img < n_images; img += gridDim.y)
    {
        const ImgDev &im = imgs[img];
        upsample_group<FMT, MINS>(samples, im, 0u, 0u, (im.width + s - 1u) / s, (im.height + s - 1u) / s, blockIdx.x * blockDim.x + threadIdx.x, pix);
    }
}

// A cropped decode (CROP): one thread per 4-pixel group of a row of each image's window crops[image].
template <int FMT, uint32_t MINS, bool CROP>
__global__ void __launch_bounds__(256)
k_upsample_libjpeg(const uint8_t *__restrict__ samples, const ImgDev *__restrict__ imgs, const CropDev *__restrict__ crops, uint32_t n_images,
                   uint8_t *__restrict__ pix)
{
    static_assert(CROP, "the whole image is k_upsample_libjpeg<FMT, MINS>");
    for (uint32_t img = blockIdx.y; img < n_images; img += gridDim.y)
    {
        const CropDev c = crops[img];
        upsample_group<FMT, MINS>(samples, imgs[img], c.x0, c.y0, c.w, c.h, blockIdx.x * blockDim.x + threadIdx.x, pix);
    }
}

// B2J_OUT_GRAY8 in the libjpeg model: libjpeg's JCS_GRAYSCALE output, the luma component's samples as they are. No
// sample plane and no second kernel: the luma blocks of the tile are transformed into a staging strip in shared memory
// behind TileSmem (the tile's MCUs side by side, MINS * yh x MINS * yv samples each, so that the *_block helpers store
// whole aligned rows), then the strip is copied into the ceil(W / s) x ceil(H / s) image.
constexpr size_t kGrayStageBytes = (size_t)kTileBlocks * 64;
static_assert(kTileSmemBytes + kGrayStageBytes <= 48 * 1024, "k_idct_gray would need its dynamic shared memory limit raised");

// `len` bytes from shared memory at src to global memory at dst (any alignment), by the lanes of one warp: the 4-byte
// words dst covers completely are stored whole, the bytes of the partial words at its ends one by one, so that the
// neighbouring bytes (another tile's, another image's) are never written.
__device__ __forceinline__ void warp_copy_out(uint8_t *__restrict__ dst, const uint8_t *src, uint32_t len, uint32_t lane)
{
    const uint32_t head = min((uint32_t)(-(uintptr_t)dst) & 3u, len);   // bytes before the first whole word
    const uint32_t words = (len - head) >> 2;
    for (uint32_t w = lane; w < words; w += 32u)
    {
        const uint8_t *p = src + head + 4u * w;
        *reinterpret_cast<uint32_t *>(dst + head + 4u * w) = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
    }
    const uint32_t tail = head + 4u * words;
    if (lane < head) dst[lane] = src[lane];
    else if (lane >= 4u && lane - 4u < len - tail) dst[tail + lane - 4u] = src[tail + lane - 4u];
}

// One launch over every tile kind. Only the luma blocks get a thread (n_mcus * yh * yv). The luma component has the largest
// factors, so jdmaster.c never doubles its DCT size: it is MINS, and each instantiation carries one transform.
// CROP: only the rows and columns inside the image's window crops[img] are copied out, to the window's pixels at the
// image's pix_off (pitch: the window's width).
template <uint32_t MINS, bool CROP>
__device__ __forceinline__ void idct_gray(const CUtensorMap &tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
                                          const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ pix, int32_t *__restrict__ status,
                                          const CropDev *__restrict__ crops)
{
    constexpr uint32_t s = 8u / MINS;
    TileSmem &sm = *tile_smem();
    uint8_t *strip = reinterpret_cast<uint8_t *>(&sm + 1);
    const uint32_t tid = threadIdx.x;
    const TileDev d = tile_load<false>(sm, &tmap, imgs, tiles, qtabs, pix, status);   // 32-bit quantisers; sd.pix = the image's output
    const uint32_t sp = sm.side.samp, n = sm.side.n_mcus;
    const uint32_t yh = sp & 15u, yv = (sp >> 4) & 15u, ny = yh * yv;
    const uint32_t tot = ny + ((sp >> 8) & 15u) * ((sp >> 12) & 15u) + ((sp >> 16) & 15u) * ((sp >> 20) & 15u);
    const uint32_t mw = yh * MINS, mh = yv * MINS, spitch = n * mw;   // an MCU's luma samples; the strip's pitch
    if (tid < n * ny)
    {
        const uint32_t m = tid / ny, k = tid % ny;   // MCU m of the tile, luma block k in it
        uint8_t *dst = strip + (k / yh) * MINS * spitch + m * mw + (k % yh) * MINS;
        const uint32_t row = m * tot + k;           // the block's row in the tile (MCU-interleaved)
        const uint32_t *q = sm.side.qt;
        if (MINS == 8u) islow_block(sm.tile, row, q, dst, spitch);
        else if (MINS == 4u) red4_block(sm.tile, row, q, dst, spitch);
        else if (MINS == 2u) red2_block(sm.tile, row, q, dst, spitch);
        else *dst = (uint8_t)islow_limit((tile_coef(sm.tile + row * 128u, row & 7u, q, 0, 0) + 4) >> 3);
    }
    __syncthreads();
    // The tile's MCUs are consecutive in raster order, so the strip holds one run of MCUs per MCU row the tile touches.
    // One warp per output row of a run; samples of padding MCUs (right of or below the output) are dropped.
    const uint32_t ow = (sm.side.width + s - 1u) / s, oh = (sm.side.height + s - 1u) / s;
    const uint32_t mcw = __ldg(&imgs[d.img].mcu_count_w), my0 = sm.side.mcu_xy[0].y;
    const uint32_t rows = (sm.side.mcu_xy[n - 1u].y - my0 + 1u) * mh;
    if constexpr (CROP)
    {
        const CropDev c = crops[d.img];   // inside the ow x oh frame (checked by the host)
        for (uint32_t i = tid >> 5; i < rows; i += kTileBlocks / 32)
        {
            const uint32_t my = my0 + i / mh, r = i % mh, y = my * mh + r;
            if (y >= c.y0 + c.h) break;
            if (y < c.y0) continue;
            const uint32_t ma = max(my * mcw, d.mcu_first) - d.mcu_first, mb = min((my + 1u) * mcw, d.mcu_first + n) - d.mcu_first;
            const uint32_t x0 = sm.side.mcu_xy[ma].x * mw, xa = max(x0, c.x0), xb = min(x0 + (mb - ma) * mw, c.x0 + c.w);
            if (xa < xb) warp_copy_out(sm.side.pix + (size_t)(y - c.y0) * c.w + (xa - c.x0), strip + r * spitch + ma * mw + (xa - x0), xb - xa, tid & 31u);
        }
    }
    else
        for (uint32_t i = tid >> 5; i < rows; i += kTileBlocks / 32)
        {
            const uint32_t my = my0 + i / mh, r = i % mh, y = my * mh + r;
            if (y >= oh) break;
            const uint32_t ma = max(my * mcw, d.mcu_first) - d.mcu_first, mb = min((my + 1u) * mcw, d.mcu_first + n) - d.mcu_first;
            const uint32_t x0 = sm.side.mcu_xy[ma].x * mw, x1 = min(x0 + (mb - ma) * mw, ow);
            if (x0 < x1) warp_copy_out(sm.side.pix + (size_t)y * ow + x0, strip + r * spitch + ma * mw, x1 - x0, tid & 31u);
        }
}

template <uint32_t MINS>
__global__ void __launch_bounds__(kTileBlocks)
k_idct_gray(const __grid_constant__ CUtensorMap tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
            const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ pix, int32_t *__restrict__ status)
{
    idct_gray<MINS, false>(tmap, imgs, tiles, qtabs, pix, status, nullptr);
}

template <uint32_t MINS, bool CROP>
__global__ void __launch_bounds__(kTileBlocks)
k_idct_gray(const __grid_constant__ CUtensorMap tmap, const ImgDev *__restrict__ imgs, const TileDev *__restrict__ tiles,
            const uint16_t *__restrict__ qtabs, uint8_t *__restrict__ pix, int32_t *__restrict__ status, const CropDev *__restrict__ crops)
{
    static_assert(CROP, "the whole image is k_idct_gray<MINS>");
    idct_gray<MINS, true>(tmap, imgs, tiles, qtabs, pix, status, crops);
}

// =====================================================================================
// Coefficient tap: int16 quantised plane -> the reference's int32 dequantised mcu_data layout.
__global__ void __launch_bounds__(256)
k_expand_coefs(const int16_t *__restrict__ coef, const uint16_t *__restrict__ qtab, uint32_t blk_count,
               uint32_t tot, uint32_t ny, uint32_t nu, int32_t *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)blk_count * 64) return;
    const uint32_t blk = (uint32_t)(i >> 6), k = (uint32_t)(i & 63);
    const uint32_t bi = blk % tot;
    const uint32_t comp = (bi >= ny ? 1u : 0u) + (bi >= ny + nu ? 1u : 0u);
    out[i] = (int32_t)coef[i] * (int32_t)qtab[comp * 64 + k];
}

// The secondary boundary (idct.h:9-18): the reference hands its device backend int32 coefficients that are already
// dequantised. They go into the int16 plane as they are (saturated: a valid 8-bit JPEG keeps them inside +-2^15) and
// the IDCT/colour kernel runs with unit quantisers.
__global__ void __launch_bounds__(256)
k_pack_coefs(const int32_t *__restrict__ in, int16_t *__restrict__ coef, size_t n_values)
{
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n_values) return;   // n_values is a multiple of 64
    const int4 v = __ldg(reinterpret_cast<const int4 *>(in + i));
    uint32_t lo, hi;
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(lo) : "r"(v.y), "r"(v.x));
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(hi) : "r"(v.w), "r"(v.z));
    *reinterpret_cast<uint2 *>(coef + i) = make_uint2(lo, hi);
}

// Output stage (SURVEY 8f rank 3, "optional resize"): box-filter reduction of the decoded pixels by an integer factor per
// axis. One thread per output sample group: BGRA / RGB24 = one output pixel (all its channels), planar RGB = one output
// sample of one plane. Every output value is the rounded mean of the input values it covers (at the right and bottom
// edges: of those that exist). blockIdx.y (strided by gridDim.y) = image.
__global__ void __launch_bounds__(256)
k_downscale(const uint8_t *__restrict__ pix, const ImgDev *__restrict__ imgs, const uint64_t *__restrict__ out_off,
            uint8_t *__restrict__ out, uint32_t n_images, uint32_t factor, int fmt)
{
    for (uint32_t img = blockIdx.y; img < n_images; img += gridDim.y)
    {
        const ImgDev &im = imgs[img];
        const uint32_t w = im.width, h = im.height, ow = (w + factor - 1) / factor, oh = (h + factor - 1) / factor;
        const uint32_t planes = fmt == B2J_OUT_RGB_PLANAR ? 3u : 1u;
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= ow * oh * planes) continue;
        const uint32_t pl = i / (ow * oh), r = i % (ow * oh), oy = r / ow, ox = r % ow;
        const uint32_t x0 = ox * factor, y0 = oy * factor, x1 = min(x0 + factor, w), y1 = min(y0 + factor, h);
        const uint32_t bpp = fmt == B2J_OUT_BGRA ? 4u : (fmt == B2J_OUT_RGB24 ? 3u : 1u);
        const uint8_t *src = pix + im.pix_off + (size_t)pl * w * h;
        uint32_t acc[4] = {0u, 0u, 0u, 0u};
        for (uint32_t y = y0; y < y1; y++)
            for (uint32_t x = x0; x < x1; x++)
            {
                const uint8_t *p = src + ((size_t)y * w + x) * bpp;
                if (bpp == 4u) { const uint32_t v = *reinterpret_cast<const uint32_t *>(p); acc[0] += v & 0xFFu; acc[1] += (v >> 8) & 0xFFu; acc[2] += (v >> 16) & 0xFFu; }
                else if (bpp == 3u) { acc[0] += p[0]; acc[1] += p[1]; acc[2] += p[2]; }
                else acc[0] += p[0];
            }
        const uint32_t n = (x1 - x0) * (y1 - y0), half = n / 2u;
        uint8_t *dst = out + out_off[img] + (size_t)pl * ow * oh + ((size_t)oy * ow + ox) * bpp;
        if (bpp == 4u)
            *reinterpret_cast<uint32_t *>(dst) = (acc[0] + half) / n | ((acc[1] + half) / n) << 8 | ((acc[2] + half) / n) << 16;
        else if (bpp == 3u) { dst[0] = (uint8_t)((acc[0] + half) / n); dst[1] = (uint8_t)((acc[1] + half) / n); dst[2] = (uint8_t)((acc[2] + half) / n); }
        else dst[0] = (uint8_t)((acc[0] + half) / n);
    }
}

// =====================================================================================
// EXIF orientation (b2j_batch_set_orientations): a copy of every image whose code is not 1, transformed. One CTA per tile
// of kOrientTile x kOrientTile source pixels of one image, from a flat host-built list over every oriented image. The
// tile's source rows are read as aligned 4-byte words into shared memory, each row keeping its misalignment; then the
// destination rows the tile covers are written as aligned words, with single bytes where a row's bytes begin or end
// inside a word. So the transposing codes 5..8 read and write whole rows too, and no byte outside an image's result is
// written: the host feed packs GRAY8 and three-byte images at 1- and 4-byte alignment. Destination (X, Y) takes the
// source pixel (x, y) with (u, v) = (Y, X) for codes 5..8, else (X, Y); x = u, or w - 1 - u for codes 2, 3, 7 and 8;
// y = v, or h - 1 - v for codes 3, 4, 6 and 7.
template <int FMT>
__global__ void __launch_bounds__(256)
k_orient(const uint8_t *__restrict__ pix, const ImgDev *__restrict__ imgs, const OrientTileDev *__restrict__ tiles, uint32_t scale,
         uint8_t *__restrict__ out)
{
    constexpr uint32_t T = kOrientTile;
    constexpr uint32_t bpp = FMT == B2J_OUT_BGRA ? 4u : (FMT == B2J_OUT_RGB24 ? 3u : 1u);
    constexpr uint32_t planes = FMT == B2J_OUT_RGB_PLANAR ? 3u : 1u;
    constexpr uint32_t pw = ((T * bpp + 3u) / 4u + 1u) | 1u;   // words per shared row: a row's bytes and its misalignment; odd,
                                                                // so that the rows of one column fall into different banks
    __shared__ uint32_t s_w[T * pw];
    const uint8_t *s_b = reinterpret_cast<const uint8_t *>(s_w);
    const OrientTileDev t = tiles[blockIdx.x];
    const ImgDev &im = imgs[t.img];
    const uint32_t w = (im.width + scale - 1u) / scale, h = (im.height + scale - 1u) / scale;
    const uint32_t code = t.tile >> 22, x0 = (t.tile & 0x7FFu) * T, y0 = ((t.tile >> 11) & 0x7FFu) * T;
    const uint32_t tw = min(T, w - x0), th = min(T, h - y0);
    const bool swap = code >= 5u, mx = code == 2u || code == 3u || code == 7u || code == 8u, my = code == 3u || code == 4u || code == 6u || code == 7u;
    const uint32_t u0 = mx ? w - x0 - tw : x0, v0 = my ? h - y0 - th : y0;   // the tile's (u, v) rectangle
    const uint32_t dx0 = swap ? v0 : u0, dy0 = swap ? u0 : v0, dw = swap ? th : tw, dh = swap ? tw : th;
    const size_t spitch = (size_t)w * bpp, dpitch = (size_t)(swap ? h : w) * bpp, plane = (size_t)w * h;
    for (uint32_t p = 0; p < planes; p++)
    {
        const uint8_t *src = pix + im.pix_off + p * plane + (size_t)y0 * spitch + x0 * bpp;
        uint8_t *dst = out + t.dst_off + p * plane + (size_t)dy0 * dpitch + dx0 * bpp;
        if (p) __syncthreads();
        for (uint32_t i = threadIdx.x; i < th * pw; i += blockDim.x)
        {
            const uint32_t r = i / pw, k = i % pw;
            const uint8_t *row = src + r * spitch;
            const uint32_t a = (uint32_t)(uintptr_t)row & 3u;
            // a whole aligned word that holds a byte of the row lies inside the plane's allocation
            if (4u * k < a + tw * bpp) s_w[r * pw + k] = __ldg(reinterpret_cast<const uint32_t *>(row - a) + k);
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < dh * pw; i += blockDim.x)
        {
            const uint32_t r = i / pw, k = i % pw, len = dw * bpp;
            uint8_t *row = dst + r * dpitch;
            const uint32_t a = (uint32_t)(uintptr_t)row & 3u;
            const int32_t b0 = (int32_t)(4u * k) - (int32_t)a;   // the word's first byte, counted from the row's first
            if (b0 >= (int32_t)len) continue;
            if constexpr (bpp == 4u)
            {
                // BGRA rows are 4-byte aligned: word k is destination pixel k
                const uint32_t uu = swap ? r : k, vv = swap ? k : r;
                const uint32_t lx = mx ? tw - 1u - uu : uu, ly = my ? th - 1u - vv : vv;
                *reinterpret_cast<uint32_t *>(row + 4u * k) = s_w[ly * pw + lx];
            }
            else
            {
                uint32_t v = 0u;
#pragma unroll
                for (uint32_t j = 0; j < 4u; j++)
                {
                    const int32_t b = b0 + (int32_t)j;
                    if (b < 0 || b >= (int32_t)len) continue;
                    const uint32_t X = (uint32_t)b / bpp, c = (uint32_t)b % bpp;
                    const uint32_t uu = swap ? r : X, vv = swap ? X : r;
                    const uint32_t lx = mx ? tw - 1u - uu : uu, ly = my ? th - 1u - vv : vv;
                    const uint32_t sa = (uint32_t)(uintptr_t)(src + ly * spitch) & 3u;
                    v |= (uint32_t)s_b[ly * pw * 4u + sa + lx * bpp + c] << (8u * j);
                }
                if (b0 >= 0 && b0 + 4 <= (int32_t)len) *reinterpret_cast<uint32_t *>(row + b0) = v;
                else
                    for (uint32_t j = 0; j < 4u; j++)
                    {
                        const int32_t b = b0 + (int32_t)j;
                        if (b >= 0 && b < (int32_t)len) row[b] = (uint8_t)(v >> (8u * j));
                    }
            }
        }
    }
}

// =====================================================================================
// Launchers (host).
size_t huff_smem_bytes(uint32_t max_lut_len) { return (size_t)kHuffThreads * 128 + kZzBytes + (size_t)max_lut_len * 2; }

cudaError_t configure_kernels(uint32_t max_lut_len)
{
    const int hb = (int)huff_smem_bytes(kLutMaxDecode);   // the decode kernels stage the decode part of a LUT set only
    cudaError_t e = cudaFuncSetAttribute(k_huff_decode<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, hb);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_huff_decode<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, hb);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_sync_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSyncSharedBytes + max_lut_len * 2));   // the walk part of a set is staged
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_sync_sweep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSyncSharedBytes + max_lut_len * 2));
}

void launch_prepass(const DecodeArgs &a, cudaStream_t s)
{
    if (a.n_chunks == 0) return;
    k_unstuff_fused<<<a.n_chunks, kScanThreads, 0, s>>>(a.raw, a.clean, a.imgs, a.chunk_img, a.chunk_state, a.clean_len, a.seg_start, a.scan_cut,
                                                              a.status);
}

void launch_huffman(const DecodeArgs &a, cudaStream_t s)
{
    if (a.n_huff_ctas == 0) return;
    k_huff_decode<false><<<a.n_huff_ctas, kHuffThreads, huff_smem_bytes(a.max_lut_dec_len), s>>>(a.clean, a.imgs, a.huff_ctas, a.seg_start, a.clean_len,
                                                                                                a.scan_cut, a.luts, a.coef, a.status, nullptr, nullptr);
}

// Streams without restart markers: chunk-wise synchronisation, the sweep, the scan, then the decode.
void launch_huffman_sync(const DecodeArgs &a, cudaStream_t s)
{
    const uint32_t n = a.n_sync_ctas, ni = a.n_sync_imgs;
    if (n == 0 || ni == 0) return;
    const size_t sync_bytes = kSyncSharedBytes + (size_t)a.max_lut_walk_len * 2;
    k_sync_chunks<<<n, kHuffThreads, sync_bytes, s>>>(a.clean, a.imgs, a.sync_ctas, a.clean_len, a.scan_cut, a.luts, a.recs, a.sync_chunk_state, a.sync_cta_base,
                                                      a.sync_stats, a.sync_use_pre ? 1u : 0u);
    k_sync_sweep<<<ni, kHuffThreads, sync_bytes, s>>>(a.clean, a.imgs, a.sync_imgs, a.clean_len, a.scan_cut, a.luts, a.recs, a.sync_chunk_state, a.sync_cta_base,
                                                     a.sync_stats);
    k_sync_cta_scan<<<ni, 32, 0, s>>>(a.imgs, a.sync_imgs, a.sync_cta_base);
    k_huff_decode<true><<<n, kHuffThreads, huff_smem_bytes(a.max_lut_dec_len), s>>>(a.clean, a.imgs, a.sync_ctas, a.seg_start, a.clean_len, a.scan_cut, a.luts,
                                                                                    a.coef, a.status, a.recs, a.sync_cta_base);
}

// The colour kernel of one output format and tile kind over `count` tiles from `first`: the narrow-quantiser
// instantiation, or the wide one when some quantiser of the batch exceeds 255.
template <int FMT, int KIND>
static void launch_idct_kind(const DecodeArgs &a, uint32_t first, uint32_t count, cudaStream_t s)
{
    if (count == 0) return;
    const auto kernel = a.any_wide_q ? k_idct_csc<false, FMT, KIND> : k_idct_csc<true, FMT, KIND>;
    kernel<<<count, kTileBlocks, kTileSmemBytes, s>>>(*a.tmap, a.imgs, a.tiles + first, a.qtabs, a.pixels, a.status);
}

template <int FMT>
static void launch_idct_format(const DecodeArgs &a, cudaStream_t s)
{
    launch_idct_kind<FMT, kTileColour>(a, 0, a.gray_tile0, s);
    launch_idct_kind<FMT, kTileGray>(a, a.gray_tile0, a.generic_tile0 - a.gray_tile0, s);
    launch_idct_kind<FMT, kTileGeneric>(a, a.generic_tile0, a.n_tiles - a.generic_tile0, s);
}

// The libjpeg model: the IDCT over every tile into the sample plane, then the upsampling / colour pass over every image.
// A cropped decode (a.crops) transforms the tiles of its crop tile list (every window has one at least) and upsamples
// the windows only.
template <int FMT, uint32_t MINS>
static void launch_libjpeg_scale(const DecodeArgs &a, cudaStream_t s)
{
    const dim3 grid((a.max_px_groups + 255u) / 256u, a.n_images < 65535u ? a.n_images : 65535u);
    if (a.crops)
    {
        k_idct_libjpeg<MINS><<<a.n_crop_tiles, kTileBlocks, kTileSmemBytes, s>>>(*a.tmap, a.imgs, a.crop_tiles, a.qtabs, a.samples, a.status);
        k_upsample_libjpeg<FMT, MINS, true><<<grid, 256, 0, s>>>(a.samples, a.imgs, a.crops, a.n_images, a.pixels);
        return;
    }
    k_idct_libjpeg<MINS><<<a.n_tiles, kTileBlocks, kTileSmemBytes, s>>>(*a.tmap, a.imgs, a.tiles, a.qtabs, a.samples, a.status);
    k_upsample_libjpeg<FMT, MINS><<<grid, 256, 0, s>>>(a.samples, a.imgs, a.n_images, a.pixels);
}

template <int FMT>
static void launch_libjpeg_format(const DecodeArgs &a, cudaStream_t s)
{
    if (a.scale == 1) launch_libjpeg_scale<FMT, 8>(a, s);   // MINS = 8 / scale, the smallest DCT size
    else if (a.scale == 2) launch_libjpeg_scale<FMT, 4>(a, s);
    else if (a.scale == 4) launch_libjpeg_scale<FMT, 2>(a, s);
    else launch_libjpeg_scale<FMT, 1>(a, s);
}

// GRAY8 in the libjpeg model: one kernel straight into the pixel plane.
template <uint32_t MINS>
static void launch_gray_scale(const DecodeArgs &a, cudaStream_t s)
{
    if (a.crops)
    {
        k_idct_gray<MINS, true><<<a.n_crop_tiles, kTileBlocks, kTileSmemBytes + kGrayStageBytes, s>>>(*a.tmap, a.imgs, a.crop_tiles, a.qtabs, a.pixels,
                                                                                                    a.status, a.crops);
        return;
    }
    k_idct_gray<MINS><<<a.n_tiles, kTileBlocks, kTileSmemBytes + kGrayStageBytes, s>>>(*a.tmap, a.imgs, a.tiles, a.qtabs, a.pixels, a.status);
}

int idct_launches(const DecodeArgs &a)
{
    if (a.n_tiles == 0) return 0;
    if (a.pixel_model == B2J_PIXELS_LIBJPEG) return a.out_format == B2J_OUT_GRAY8 ? 1 : 2;
    return (a.gray_tile0 > 0 ? 1 : 0) + (a.generic_tile0 > a.gray_tile0 ? 1 : 0) + (a.n_tiles > a.generic_tile0 ? 1 : 0);
}

void launch_idct(const DecodeArgs &a, cudaStream_t s)
{
    if (a.pixel_model == B2J_PIXELS_LIBJPEG)
    {
        if (a.n_tiles == 0) return;
        if (a.out_format == B2J_OUT_GRAY8)
        {
            if (a.scale == 1) launch_gray_scale<8>(a, s);   // MINS = 8 / scale
            else if (a.scale == 2) launch_gray_scale<4>(a, s);
            else if (a.scale == 4) launch_gray_scale<2>(a, s);
            else launch_gray_scale<1>(a, s);
        }
        else if (a.out_format == B2J_OUT_RGB24) launch_libjpeg_format<B2J_OUT_RGB24>(a, s);
        else if (a.out_format == B2J_OUT_RGB_PLANAR) launch_libjpeg_format<B2J_OUT_RGB_PLANAR>(a, s);
        else launch_libjpeg_format<B2J_OUT_BGRA>(a, s);
        return;
    }
    if (a.out_format == B2J_OUT_RGB24) launch_idct_format<B2J_OUT_RGB24>(a, s);
    else if (a.out_format == B2J_OUT_RGB_PLANAR) launch_idct_format<B2J_OUT_RGB_PLANAR>(a, s);
    else launch_idct_format<B2J_OUT_BGRA>(a, s);
}

void launch_downscale(const uint8_t *pix, const ImgDev *imgs, const uint64_t *out_off, uint8_t *out, uint32_t n_images, uint32_t max_out_samples,
                      uint32_t factor, int fmt, cudaStream_t s)
{
    if (n_images == 0 || max_out_samples == 0) return;
    const dim3 grid((max_out_samples + 255u) / 256u, n_images < 65535u ? n_images : 65535u);   // gridDim.y is at most 65535
    k_downscale<<<grid, 256, 0, s>>>(pix, imgs, out_off, out, n_images, factor, fmt);
}

void launch_orient(const uint8_t *pix, const ImgDev *imgs, const OrientTileDev *tiles, uint32_t n_tiles, uint32_t scale, int fmt, uint8_t *out,
                   cudaStream_t s)
{
    if (n_tiles == 0) return;   // one CTA per tile: a flat grid, so any number of images fits
    if (fmt == B2J_OUT_RGB24) k_orient<B2J_OUT_RGB24><<<n_tiles, 256, 0, s>>>(pix, imgs, tiles, scale, out);
    else if (fmt == B2J_OUT_RGB_PLANAR) k_orient<B2J_OUT_RGB_PLANAR><<<n_tiles, 256, 0, s>>>(pix, imgs, tiles, scale, out);
    else if (fmt == B2J_OUT_GRAY8) k_orient<B2J_OUT_GRAY8><<<n_tiles, 256, 0, s>>>(pix, imgs, tiles, scale, out);
    else k_orient<B2J_OUT_BGRA><<<n_tiles, 256, 0, s>>>(pix, imgs, tiles, scale, out);
}

void launch_pack(const int32_t *in, int16_t *coef, size_t n_values, cudaStream_t s)
{
    if (n_values == 0) return;
    const size_t threads = (n_values + 3) / 4;
    k_pack_coefs<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(in, coef, n_values);
}

void launch_expand(const int16_t *coef, const uint16_t *qtab, uint32_t blk_count, uint32_t tot, uint32_t ny, uint32_t nu, int32_t *out, cudaStream_t s)
{
    const size_t n = (size_t)blk_count * 64;
    if (!n) return;
    k_expand_coefs<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(coef, qtab, blk_count, tot, ny, nu, out);
}

} // namespace b2j
