// host_parse.cpp -- header parsing from memory (host side of the boundary).
//
// Restates what the reference's load_jpg() does before it reaches the scan data
// (parser.cpp:272-372) together with its segment readers (parser.cpp:7-270), the accept gate
// is_supported_file() (decoder.cpp:18-70) and the geometry part of decode_init()
// (decoder.cpp:161-199), for a file held in memory. Accept/reject behaviour follows the
// reference (only APPn directly behind SOI are skipped; any marker other than DQT/SOF0/DHT/DRI/SOS
// ends parsing; SOF0 with 3 components of 8 bits; one 3-component scan with Ss,Se,AhAl =
// 0,63,0). Deviation, documented in DESIGN.md: Huffman table ids above 3 are refused (the
// reference keeps 16 DC + 16 AC slots, parser.cpp:176).
#include "b2j_internal.h"

#include <string.h>

namespace {

struct Reader
{
    const uint8_t *p;
    size_t len, pos;
    bool take(void *dst, size_t n)
    {
        if (n > len - pos) return false;
        if (dst) memcpy(dst, p + pos, n);
        pos += n;
        return true;
    }
};

inline unsigned be16(const uint8_t *b) { return ((unsigned)b[0] << 8) | b[1]; }

// parser.cpp:47-100
bool parse_dqt(b2j_image_desc &d, Reader &r, size_t len, bool robust)
{
    while (len > 0)
    {
        uint8_t head, raw[128];
        if (!r.take(&head, 1)) return false;
        const int prec = head >> 4, id = head & 0xF;
        if (id > 3 || (d.quant_present[id] && !robust) || prec > 1) return false;   // robust: a later DQT redefines the slot
        const size_t body = prec ? 128 : 64;
        if (!r.take(raw, body)) return false;
        for (int i = 0; i < 64; i++)
            d.quant[id][i] = !prec ? raw[i]
                             : robust ? (uint16_t)((raw[2 * i] << 8) | raw[2 * i + 1])     // big-endian, ITU T.81 B.2.4.1
                                      : (uint16_t)(raw[2 * i] | (raw[2 * i + 1] << 8));    // no byte swap: parser.cpp:81-87
        d.quant_present[id] = 1;
        if (len < body + 1) return false;
        len -= body + 1;
    }
    return true;
}

// parser.cpp:102-130
bool parse_sof0(b2j_image_desc &d, Reader &r, size_t len, bool allow_gray)
{
    uint8_t b[15];
    if (allow_gray && len == 9)
    {
        // one-component frame (B2J_GATE_GRAY): a single 1x1-sampled component
        if (!r.take(b, 9) || b[0] != 8 || b[5] != 1 || b[7] != 0x11) return false;
        d.height = (int32_t)be16(b + 1);
        d.width = (int32_t)be16(b + 3);
        d.sampling[0] = 0x11; d.sampling[1] = d.sampling[2] = 0;
        d.quant_id[0] = d.quant_id[1] = d.quant_id[2] = b[8];
        d.color_space = B2J_CS_GRAY;
        return true;
    }
    if (len != sizeof(b) || !r.take(b, sizeof(b))) return false;
    if (b[0] != 8 || b[5] != 3) return false;
    d.height = (int32_t)be16(b + 1);
    d.width = (int32_t)be16(b + 3);
    for (int c = 0; c < 3; c++)
    {
        d.sampling[c] = b[6 + 3 * c + 1];
        d.quant_id[c] = b[6 + 3 * c + 2];
    }
    return true;
}

// parser.cpp:170-270
bool parse_dht(b2j_image_desc &d, Reader &r, size_t len, bool robust)
{
    while (len > 0)
    {
        uint8_t head, counts[16];
        if (!r.take(&head, 1)) return false;
        const int tc = head >> 4, th = head & 0xF;
        if (tc > 1 || th > 3) return false;
        const int slot = tc * 4 + th;
        if (d.huff_present[slot] && !robust) return false;
        if (!r.take(counts, 16)) return false;
        memset(d.huff_counts[slot], 0, 16);
        unsigned total = 0, code = 0;
        for (int l = 1; l <= 16; l++)
        {
            total += counts[l - 1];
            code += counts[l - 1];
            if (counts[l - 1] && ((code - 1) >> l)) return false;   // code space exhausted: parser.cpp:239
            code <<= 1;
        }
        if (total > 256) return false;
        memcpy(d.huff_counts[slot], counts, 16);
        if (total && !r.take(d.huff_symbols[slot], total)) return false;
        d.huff_present[slot] = 1;
        if (len < 17u + total) return false;
        len -= 17u + total;
    }
    return true;
}

// parser.cpp:132-154
bool parse_sos(b2j_image_desc &d, Reader &r, size_t len)
{
    uint8_t b[10];
    if (d.color_space == B2J_CS_GRAY)
    {
        if (len != 6 || !r.take(b, 6)) return false;
        if (b[0] != 1 || b[3] != 0 || b[4] != 0x3F || b[5] != 0) return false;
        d.huff_id[0] = d.huff_id[1] = d.huff_id[2] = b[2];
        return true;
    }
    if (len != sizeof(b) || !r.take(b, sizeof(b))) return false;
    if (b[0] != 3 || b[7] != 0 || b[8] != 0x3F || b[9] != 0) return false;
    for (int c = 0; c < 3; c++) d.huff_id[c] = b[1 + 2 * c + 1];
    return true;
}

// decoder.cpp:18-70
int check_gate(const b2j_image_desc &d, int gate)
{
    if (d.width <= 0 || d.height <= 0) return B2J_E_UNSUPPORTED;
    for (int c = 0; c < 3; c++)
        if (d.quant_id[c] > 3 || !d.quant_present[d.quant_id[c]]) return B2J_E_UNSUPPORTED;
    for (int c = 0; c < 3; c++)
    {
        const int td = d.huff_id[c] >> 4, ta = d.huff_id[c] & 0xF;
        if (td > 3 || ta > 3 || !d.huff_present[td] || !d.huff_present[4 + ta]) return B2J_E_UNSUPPORTED;
    }
    // the decode kernels hold an image's decode tables in shared memory: tables whose two-level decode tables do not
    // fit together (three components with tables of 256 codes up to 16 bits long) are refused here, per file, rather
    // than when the batch that holds the file is built (documented deviation, include/b2j.h)
    if (b2j::lut_set_decode_entries(d) > (size_t)b2j::kLutMaxDecode) return B2J_E_UNSUPPORTED;
    if (d.color_space == B2J_CS_GRAY) return B2J_OK;   // admitted by parse_sof0 under B2J_GATE_GRAY only
    const int y = d.sampling[0];
    if (d.sampling[1] == 0x11 && d.sampling[2] == 0x11 && (y == 0x22 || y == 0x11)) return B2J_OK;   // decoder.cpp:58-69
    if (gate != B2J_GATE_EXTENDED) return B2J_E_UNSUPPORTED;
    // extended: any luma sampling with chroma factors that divide it, at most 10 blocks per MCU (ITU T.81 B.2.3)
    const int yh = y >> 4, yv = y & 0xF;
    if (yh < 1 || yh > 4 || yv < 1 || yv > 4) return B2J_E_UNSUPPORTED;
    int tot = yh * yv;
    for (int c = 1; c < 3; c++)
    {
        const int h = d.sampling[c] >> 4, v = d.sampling[c] & 0xF;
        if (h < 1 || v < 1 || yh % h || yv % v) return B2J_E_UNSUPPORTED;
        tot += h * v;
    }
    return tot <= 10 ? B2J_OK : B2J_E_UNSUPPORTED;
}

// decoder.cpp:161-192
void derive_geometry(b2j_image_desc &d)
{
    int mh = 0, mv = 0;
    d.tot_blks_per_mcu = 0;
    for (int c = 0; c < 3; c++)
    {
        const int h = d.sampling[c] >> 4, v = d.sampling[c] & 0xF;
        if (h > mh) mh = h;
        if (v > mv) mv = v;
        d.blks_per_mcu[c] = h * v;
        d.tot_blks_per_mcu += h * v;
    }
    d.mcu_width = 8 * mh;
    d.mcu_height = 8 * mv;
    d.mcu_count_w = (d.width - 1) / d.mcu_width + 1;
    d.mcu_count_h = (d.height - 1) / d.mcu_height + 1;
    d.mcu_count = d.mcu_count_w * d.mcu_count_h;
    d.blk_count = d.mcu_count * d.tot_blks_per_mcu;
    if (d.color_space != B2J_CS_GRAY)
        d.color_space = d.sampling[0] == 0x22 ? B2J_CS_YUV411 : (d.sampling[0] == 0x11 ? B2J_CS_YUV444 : B2J_CS_OTHER);
}

} // namespace

extern "C" int b2j_parse_header(const uint8_t *file, size_t len, int gate_flags, b2j_image_desc *out)
{
    if (!file || !out) return B2J_E_ARG;
    const bool robust = (gate_flags & B2J_PARSE_ROBUST) != 0;
    const int gate = gate_flags & 1;
    const bool allow_gray = (gate_flags & B2J_GATE_GRAY) != 0;
    b2j_image_desc &d = *out;
    memset(&d, 0, sizeof(d));
    Reader r{file, len, 0};
    uint8_t tag[2], lb[2];
    if (!r.take(tag, 2) || tag[0] != 0xFF || tag[1] != 0xD8) return B2J_E_FORMAT;
    // APPn directly after SOI (parser.cpp:295-322); only the second tag byte is examined
    tag[1] = 0;
    while (r.take(tag, 2) && tag[1] >= 0xE0 && tag[1] <= 0xEF)
    {
        if (!r.take(lb, 2)) return B2J_E_FORMAT;
        const size_t l = be16(lb);
        if (l < 2 || !r.take(nullptr, l - 2)) return B2J_E_FORMAT;
        tag[1] = 0;
    }
    while (tag[1] != 0)
    {
        if (robust)
        {
            // resynchronise on FF, skip fill bytes, stand-alone markers and anything length-prefixed we do not need
            while (tag[0] != 0xFF || tag[1] == 0xFF || tag[1] == 0x00)
            {
                tag[0] = tag[1];
                if (!r.take(&tag[1], 1)) return B2J_E_FORMAT;
            }
            const uint8_t m = tag[1];
            const bool needed = m == 0xDB || m == 0xC0 || m == 0xC4 || m == 0xDD || m == 0xDA;
            if (m == 0xD9) return B2J_E_FORMAT;
            if ((m >= 0xC1 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC)) return B2J_E_UNSUPPORTED;   // not baseline
            if (!needed)
            {
                if ((m >= 0xD0 && m <= 0xD7) || m == 0x01) { if (!r.take(tag, 2)) return B2J_E_FORMAT; continue; }
                if (!r.take(lb, 2)) return B2J_E_FORMAT;
                const size_t l = be16(lb);
                if (l < 2 || !r.take(nullptr, l - 2) || !r.take(tag, 2)) return B2J_E_FORMAT;
                continue;
            }
        }
        if (!r.take(lb, 2)) return B2J_E_FORMAT;
        const size_t seglen = (uint16_t)(be16(lb) - 2);
        switch (tag[1])
        {
        case 0xDB: if (!parse_dqt(d, r, seglen, robust)) return B2J_E_FORMAT; break;
        case 0xC0: if (!parse_sof0(d, r, seglen, allow_gray)) return B2J_E_FORMAT; break;
        case 0xC4: if (!parse_dht(d, r, seglen, robust)) return B2J_E_FORMAT; break;
        case 0xDD:
            if (seglen != 2 || !r.take(lb, 2)) return B2J_E_FORMAT;   // parser.cpp:156-168
            d.restart_interval = (int32_t)be16(lb);
            break;
        case 0xDA:
        {
            if (!parse_sos(d, r, seglen)) return B2J_E_FORMAT;
            const int rc = check_gate(d, gate);
            if (rc != B2J_OK) return rc;
            derive_geometry(d);
            d.scan_offset = r.pos;
            d.scan_size = len - r.pos;
            // a file that ends right behind the SOS header has no entropy-coded data at all: the reference gives up
            // on it with "data incomplete" (decoder.cpp:310-314)
            return d.scan_size ? B2J_OK : B2J_E_DATA;
        }
        default:   // SOF1..3 (parser.cpp:347-352), EOI, COM, late APPn: the reference stops here
            return tag[1] >= 0xC1 && tag[1] <= 0xC3 ? B2J_E_UNSUPPORTED : B2J_E_FORMAT;
        }
        if (!r.take(tag, 2)) return B2J_E_FORMAT;
    }
    return B2J_E_FORMAT;
}
