// b2j_internal.h -- data layout shared by the host runtime and the kernels (not part of the ABI).
#ifndef B2J_INTERNAL_H_INCLUDED
#define B2J_INTERNAL_H_INCLUDED

#include <stdint.h>
#include <stddef.h>
#include <vector>

#include "../../include/b2j.h"

namespace b2j {

// ---------------------------------------------------------------- constants ------------
constexpr int kScanGroups = 4;           // 16-byte groups per thread in the pre-pass (4 loads in flight per thread)
constexpr int kScanThreads = 256;
constexpr int kScanChunkBytes = kScanThreads * kScanGroups * 16;   // bytes of raw scan one CTA of the pre-pass handles
constexpr int kHuffThreads = 128;        // decode lanes (= segments) per Huffman CTA
constexpr int kSubBytes = 128;           // self-synchronising decode: bytes of clean stream per sub-sequence (one lane each); 64 and 32 were measured slower (DESIGN.md)
constexpr int kSyncPre = 2;              // chunk-wise synchronisation (b2j_sync.h): sub-sequences walked in front of a chunk
constexpr int kSyncLanes = kHuffThreads - kSyncPre;   // output sub-sequences per chunk
constexpr int kLutBits = 10;             // primary Huffman LUT width, AC tables (one lookup per coefficient)
constexpr int kLutBitsDc = 6;            // DC tables (one lookup per block): small, the shared memory goes to the stream rings
constexpr int kLutHeader = 16;           // u16 words of header in front of a LUT set:
                                         //   [0..2] DC table of component c, [3..5] AC table (decode tables, entry format below)
                                         //   [6..8] DC walk table, [9..11] AC walk table (self-synchronisation walks, b2j_sync.h)
                                         //   [12]   length of the decode part of the set (header + decode tables), a multiple of 8
constexpr int kLutMaxDecode = 12288;     // u16 entries of the decode part of a LUT set (24 KB of shared memory)
constexpr int kLutMaxEntries = 32768;    // u16 entries of a whole LUT set, walk tables included (64 KB)
constexpr int kWalkBits = 10;            // index width of the AC walk tables (several AC symbols per lookup)
constexpr int kWalkBitsDc = 8;           // index width of the DC walk tables: small, shared memory decides how many CTAs an SM holds
constexpr int kTileBlocks = 192;         // 8x8 blocks per IDCT/colour tile (= threads per CTA)
constexpr uint32_t kSegInvalid = 0xFFFFFFFFu;
constexpr uint32_t kChunkDead = 0xFFFFFFFFu;
constexpr uint32_t kNoTerm = 0xFFFFu;

// LUT entry (u16):
//   leaf    : bits 0-4  = code length (1..16), bit 5 = 1
//             AC tables: bits 6-9 = value-bit count (size nibble), bits 10-15 = zero run (0..15); the
//                        end-of-block symbol 0x00 carries run kRunEob = 63, so that it ends the block through
//                        the ordinary "position >= 64" test of the decode loop
//             DC tables: bits 6-10 = value-bit count (category 0..16)
//   escape  : bits 0-5  = extra index bits nb (1..16 - primary width, i.e. < 32: bit 5 clear), bits 6-15 = sub-table
//             offset relative to the end of the primary table, in units of kLutSubAlign entries
//   invalid : 0 (no codeword has this prefix)
// Walk tables, used by the walks of the self-synchronising path only (they need no coefficient values): 32-bit
// entries indexed by the next kWalkBits (AC) / kWalkBitsDc (DC) bits, two 16-bit halves of one layout:
//          bits 0-4  bits consumed (codes + value bits, <= 31)
//          bit  7    the set ends with the end-of-block symbol
//          bits 8-15 scan positions needed: sum of run + 1, plus 1 for a closing end-of-block symbol (the block must
//                    not be complete in front of it); <= 64; 0xFF = no entry
//   AC : the symbols whose CODES lie completely inside the index, up to and including an end-of-block, form a group.
//        Low half = the group, high half = its first symbol alone. The group is taken where position + (bits 8-15)
//        <= 64 (a block that fills up without an end-of-block code ends inside a group: then the first symbol is
//        taken alone); the block is complete behind a set when its bit 7 is set or the position reaches 64.
//   DC : low half = the symbol where code + value bits fit into the index (bits consumed = code length + category,
//        positions = 1), high half = the DC difference itself (int16).
//   bits 8-15 of the low half above 64 mark the special entries:
//   0xFE (AC) : escape -- the code is longer than the index: bits 0-4 = further index bits nb, bits 16-31 = position of
//               a sub-table of 1 << nb one-symbol entries (both halves alike), counted in entries from the table start
//   0xFD (DC) : the value bits reach past the index: bits 0-4 = code length, bits 16-20 = category
//   0xFF      : no entry (kWalkNoEntry): one symbol through the decode tables (DC code longer than the index) or no codeword
constexpr uint32_t kWalkNoEntry = 0xFF00FF00u;
constexpr uint32_t kWalkEscape = 0xFEu, kWalkDcWide = 0xFDu;
constexpr uint32_t kRunEob = 63;
constexpr uint32_t kLutSubAlign = 8;     // sub-tables start on multiples of 8 entries behind the primary table

// sampling layouts the colour kernel knows (luma h x v with 1x1 chroma)
enum SamplingMode : uint32_t { kMode444 = 0, kMode420 = 1, kMode422 = 2, kMode440 = 3, kModeGray = 4, kModeGeneric = 5 };   // gray: one component; generic: any other layout

// Per-image record in device memory.
struct ImgDev
{
    uint64_t raw_off;      // byte offset of the scan in raw[] and of the clean stream in clean[] (16 B aligned)
    uint64_t pix_off;      // byte offset of the BGRA image in pixels[] (256 B aligned)
    uint32_t raw_len;      // entropy-coded bytes (to the end of the file)
    uint32_t chunk_first;  // first pre-pass chunk of this image
    uint32_t n_chunks;
    uint32_t seg_first;    // first decode segment (restart interval) of this image
    uint32_t n_segs;
    uint32_t blk_first;    // first row of this image in the coefficient plane
    uint32_t blk_count;
    uint32_t mcu_count;
    uint32_t mcu_count_w;
    uint32_t restart_interval; // MCUs per segment (== mcu_count when the file has no DRI)
    uint32_t has_dri;
    uint32_t width, height;
    uint32_t lut_off;      // u16 offset of the LUT set in luts[]
    uint32_t lut_len;      // u16 length of the LUT set (header, decode tables, walk tables)
    uint32_t lut_dec_len;  // u16 length of its decode part (what k_huff_decode stages)
    uint32_t mode;         // SamplingMode
    uint32_t tot_blks;     // blocks per MCU
    uint32_t ny_blks;      // luma blocks per MCU
    uint32_t nu_blks;      // blocks of the second component per MCU
    uint32_t samp;         // sampling factors, one nibble each: yh | yv<<4 | uh<<8 | uv<<12 | vh<<16 | vv<<20
    uint32_t yh;           // luma blocks per MCU row
    uint32_t wide_q;       // 1 when some quantiser value exceeds 255
    uint32_t sub_first;    // self-synchronising path (streams without DRI): first sub-sequence record of this image
    uint32_t n_sub_max;    // upper bound of its sub-sequence count (from raw_len); 0 = restart-interval path
    uint32_t scta_first;   // its first decode CTA on the self-synchronising path
};

// Self-synchronising decode, one record per sub-sequence j of kSubBytes*8 bits of clean stream:
// the decoder state when it leaves the sub-sequence (the first symbol that STARTS at or behind the
// end of the sub-sequence is not decoded), and what was met inside it.
struct SubRec
{
    uint32_t p;         // bit position of the exit state (>= end of the sub-sequence)
    uint32_t cz;        // block-in-MCU index | zig-zag position << 8 (0 = next symbol is a DC code); kSubInvalid = no valid state
    uint32_t nblk;      // blocks whose DC code starts inside the sub-sequence
    int32_t dc[3];      // sum of the DC differences of those blocks, per component
    uint32_t fs;        // bit position of the first of those blocks (kSubNone: none)
    uint32_t fc;        // its block-in-MCU index
};
// Checkpoint of round 0 at the middle of a sub-sequence, same layout as SubRec: p / cz = the state at the first
// symbol at or behind the middle, the other fields = what the second half contributes.
struct SubMid { uint32_t p, cz, nblk; int32_t dc[3]; uint32_t fs, fc; };
struct SubPre { uint32_t blk; int32_t dc[3]; };   // exclusive prefix over the sub-sequences of one image (formed inside the decode CTA)
constexpr uint32_t kSubInvalid = 0xFFFFFFFFu;
constexpr uint32_t kSubNone = 0xFFFFFFFFu;

struct HuffCtaDev { uint32_t img; uint32_t seg_first; };   // segment index local to the image
// One IDCT/colour tile: up to kTileBlocks consecutive blocks (whole MCUs) of one image.
struct TileDev
{
    uint32_t img;
    uint32_t mcu_first;   // first MCU of the tile inside the image
    uint32_t row_first;   // first row of the tile in the coefficient plane (the TMA y coordinate)
    uint32_t info;        // SamplingMode | n_mcus << 8
};

// ---------------------------------------------------------------- host helpers ---------
// Canonical Huffman table -> two-level LUT. Returns false when the table cannot be built
// (code space overflow) or needs more than `max_entries` entries.
bool build_huff_lut(const uint8_t counts[16], const uint8_t *symbols, bool is_dc, std::vector<uint16_t> &out, size_t max_entries);

// Entries build_huff_lut() makes for this table (no limit applied).
size_t huff_lut_entries(const uint8_t counts[16], bool is_dc);

// Entries of the decode part of an image's LUT set (header + the decode tables of its distinct table slots), the
// part that must fit kLutMaxDecode.
size_t lut_set_decode_entries(const b2j_image_desc &d);

// Canonical Huffman table -> walk table (1 << kWalkBits 32-bit entries as pairs of u16, format above).
bool build_walk_lut(const uint8_t counts[16], const uint8_t *symbols, bool is_dc, std::vector<uint16_t> &out);

// LUT set for one image: header (offsets of the DC/AC table of each component) + tables.
bool build_lut_set(const b2j_image_desc &d, std::vector<uint16_t> &out);

} // namespace b2j
#endif
