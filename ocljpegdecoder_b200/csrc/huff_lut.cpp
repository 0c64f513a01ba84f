// huff_lut.cpp -- host-side construction of the Huffman decode tables the kernels use.
//
// The reference decodes with a 16-ary trie walked 4 bits at a time (huffman.h:200-314, built at
// decoder.cpp:266-273 from the ASCII code strings of parser.cpp:221-257). On the GPU a symbol is
// one shared-memory lookup: the next kLutBits bits index a primary table whose entry carries
// code length, value-bit count and zero run; the rare longer codes take one more lookup in a
// sub-table addressed by the remaining bits. Both are prefix-code decoders of the same canonical
// code, so they accept and reject exactly the same bit strings.
#include "b2j_internal.h"

#include <string.h>

namespace b2j {

namespace {
inline uint16_t leaf_entry(int len, int sym, bool is_dc)
{
    if (is_dc)
    {
        if (sym > 16) return 0;   // category > 16: not decodable here
        return (uint16_t)(len | 32 | (sym << 6));
    }
    const int size = sym & 15, run = sym == 0 ? (int)kRunEob : (sym >> 4);
    return (uint16_t)(len | 32 | (size << 6) | (run << 10));
}
} // namespace

bool build_huff_lut(const uint8_t counts[16], const uint8_t *symbols, bool is_dc, std::vector<uint16_t> &out, size_t max_entries)
{
    const int K = is_dc ? kLutBitsDc : kLutBits;
    struct Code { uint32_t code; int len; int sym; };
    Code codes[256];
    int n = 0;
    uint32_t code = 0;
    for (int l = 1; l <= 16; l++)
    {
        for (int i = 0; i < counts[l - 1]; i++)
        {
            if (n >= 256 || (code >> l)) return false;   // parser.cpp:239 "invalid tree"
            codes[n].code = code; codes[n].len = l; codes[n].sym = symbols[n];
            n++; code++;
        }
        code <<= 1;
    }
    out.assign((size_t)1 << K, 0);
    // longest code below each K-bit prefix
    std::vector<uint8_t> maxlen((size_t)1 << K, 0);
    for (int i = 0; i < n; i++)
    {
        const Code &c = codes[i];
        if (c.len <= K)
        {
            const uint32_t first = c.code << (K - c.len), cnt = 1u << (K - c.len);
            const uint16_t e = leaf_entry(c.len, c.sym, is_dc);
            for (uint32_t k = 0; k < cnt; k++) out[first + k] = e;
        }
        else
        {
            const uint32_t prefix = c.code >> (c.len - K);
            if (maxlen[prefix] < c.len) maxlen[prefix] = (uint8_t)c.len;
        }
    }
    // one sub-table per prefix that has long codes
    std::vector<uint32_t> sub_off((size_t)1 << K, 0);
    for (uint32_t p = 0; p < (1u << K); p++)
    {
        if (!maxlen[p]) continue;
        const int nb = maxlen[p] - K;
        while ((out.size() - ((size_t)1 << K)) % kLutSubAlign) out.push_back(0);   // escapes address sub-tables in units of kLutSubAlign
        const size_t rel = out.size() - ((size_t)1 << K);
        if (rel / kLutSubAlign >= 1024) return false;
        sub_off[p] = (uint32_t)out.size();
        out[p] = (uint16_t)(nb | ((rel / kLutSubAlign) << 6));
        out.resize(out.size() + ((size_t)1 << nb), 0);
        if (out.size() > max_entries) return false;
    }
    for (int i = 0; i < n; i++)
    {
        const Code &c = codes[i];
        if (c.len <= K) continue;
        const uint32_t prefix = c.code >> (c.len - K);
        const int nb = maxlen[prefix] - K, extra = c.len - K;
        const uint32_t rem = c.code & ((1u << extra) - 1u);
        const uint32_t first = rem << (nb - extra), cnt = 1u << (nb - extra);
        const uint16_t e = leaf_entry(c.len, c.sym, is_dc);
        for (uint32_t k = 0; k < cnt; k++) out[sub_off[prefix] + first + k] = e;
    }
    return out.size() <= max_entries;
}

size_t huff_lut_entries(const uint8_t counts[16], bool is_dc)
{
    // what build_huff_lut() builds, counted: canonical codes come in increasing order, so the primary prefixes with long
    // codes come in increasing order too, and the last code below a prefix is its longest
    const int K = is_dc ? kLutBitsDc : kLutBits;
    size_t rel = 0;
    uint32_t code = 0, prefix = 0;
    int longest = 0;
    auto close = [&]() {
        if (!longest) return;
        while (rel % kLutSubAlign) rel++;
        rel += (size_t)1 << (longest - K);
    };
    for (int l = 1; l <= 16; l++)
    {
        for (int i = 0; i < counts[l - 1]; i++, code++)
        {
            if (l <= K) continue;
            const uint32_t p = code >> (l - K);
            if (longest && p != prefix) close();
            prefix = p;
            longest = l;
        }
        code <<= 1;
    }
    close();
    return ((size_t)1 << K) + rel;
}

size_t lut_set_decode_entries(const b2j_image_desc &d)
{
    // build_lut_set(): the header, then one decode table per distinct table slot, padded to 16 bytes
    size_t n = kLutHeader;
    bool seen[8] = {false, false, false, false, false, false, false, false};
    for (int c = 0; c < 3; c++)
        for (int kind = 0; kind < 2; kind++)
        {
            const int th = kind == 0 ? (d.huff_id[c] >> 4) : (d.huff_id[c] & 0xF);
            if (th > 3) continue;
            const int slot = kind * 4 + th;
            if (seen[slot]) continue;
            seen[slot] = true;
            n += huff_lut_entries(d.huff_counts[slot], kind == 0);
        }
    return (n + 7) & ~(size_t)7;
}

bool build_walk_lut(const uint8_t counts[16], const uint8_t *symbols, bool is_dc, std::vector<uint16_t> &out)
{
    const int K = is_dc ? kWalkBitsDc : kWalkBits;
    struct Code { uint32_t code; int len; int sym; };
    Code codes[256];
    int n = 0;
    uint32_t code = 0;
    for (int l = 1; l <= 16; l++)
    {
        for (int i = 0; i < counts[l - 1]; i++)
        {
            if (n >= 256 || (code >> l)) return false;
            codes[n].code = code; codes[n].len = l; codes[n].sym = symbols[n];
            n++; code++;
        }
        code <<= 1;
    }
    // the codeword (if any) that starts at bit `pos` of the K-bit window w and ends inside it
    auto match = [&](uint32_t w, int pos) -> const Code * {
        for (int i = 0; i < n; i++)
        {
            const Code &c = codes[i];
            if (c.len > K - pos) break;   // canonical order: lengths never decrease
            if (((w >> (K - pos - c.len)) & ((1u << c.len) - 1u)) == c.code) return &c;
        }
        return nullptr;
    };
    auto put = [&](size_t w, uint32_t v) { out[2 * w] = (uint16_t)v; out[2 * w + 1] = (uint16_t)(v >> 16); };
    // 32-bit entries, stored as two u16 each (little endian)
    out.assign((size_t)2 << K, 0);
    for (uint32_t w = 0; w < (1u << K); w++) put(w, kWalkNoEntry);
    if (is_dc)
    {
        for (uint32_t w = 0; w < (1u << K); w++)
        {
            const Code *c = match(w, 0);
            if (!c || c->sym > 16) continue;
            const int size = c->sym;
            if (c->len + size > K)
            {
                // the value bits reach past the index: the walk extracts them itself
                put(w, (uint32_t)c->len | kWalkDcWide << 8 | (uint32_t)size << 16);
                continue;
            }
            // code and value bits inside the index: the entry carries the difference (decoder.cpp:72-82)
            const uint32_t v = size ? (w >> (K - c->len - size)) & ((1u << size) - 1u) : 0u;
            const int32_t diff = size == 0 ? 0 : ((v >> (size - 1)) ? (int32_t)v : (int32_t)v + 1 - (1 << size));
            put(w, (uint32_t)(c->len + size) | 1u << 8 | (uint32_t)(uint16_t)(int16_t)diff << 16);
        }
        return true;
    }
    auto single = [&](const Code &c) -> uint32_t {
        const uint32_t e = c.sym == 0x00 ? 1u : 0u;
        const uint32_t adv = e ? 1u : (uint32_t)(c.sym >> 4) + 1u, bits = (uint32_t)c.len + (e ? 0u : (uint32_t)(c.sym & 15));
        const uint32_t half = bits | e << 7 | adv << 8;
        return half | half << 16;
    };
    for (uint32_t w = 0; w < (1u << K); w++)
    {
        int pos = 0, zadv = 0, nsym = 0, nbits = 0, eob = 0;
        uint32_t first = 0;
        while (pos < K)
        {
            const Code *c = match(w, pos);
            if (!c) break;
            int adv, bits, e = 0;
            if (c->sym == 0x00) { adv = 0; bits = c->len; e = 1; }   // end of block (decoder.cpp:247-249)
            else
            {
                adv = (c->sym >> 4) + 1;   // a coefficient behind `run` zeros, or run + 1 zeros when size == 0 (decoder.cpp:250-256)
                bits = c->len + (c->sym & 15);
            }
            if (zadv + adv + e > 64 || pos + bits > 31) break;
            zadv += adv; pos += bits; nbits = pos; eob = e; nsym++;
            if (nsym == 1) first = (uint32_t)nbits | (uint32_t)eob << 7 | (uint32_t)(zadv + eob) << 8;
            if (e) break;
        }
        if (!nsym) continue;
        const uint32_t group = (uint32_t)nbits | (uint32_t)eob << 7 | (uint32_t)(zadv + eob) << 8;
        put(w, group | first << 16);
    }
    // codes longer than the index: one sub-table per K-bit prefix, behind the primary table (one symbol per entry)
    std::vector<uint8_t> maxlen((size_t)1 << K, 0);
    for (int i = 0; i < n; i++)
        if (codes[i].len > K)
        {
            const uint32_t prefix = codes[i].code >> (codes[i].len - K);
            if (maxlen[prefix] < codes[i].len) maxlen[prefix] = (uint8_t)codes[i].len;
        }
    std::vector<uint32_t> sub_at((size_t)1 << K, 0);
    for (uint32_t pfx = 0; pfx < (1u << K); pfx++)
    {
        if (!maxlen[pfx]) continue;
        const int nb = maxlen[pfx] - K;
        const size_t at = out.size() / 2;
        if (at >= 0x10000) return false;
        sub_at[pfx] = (uint32_t)at;
        put(pfx, (uint32_t)nb | kWalkEscape << 8 | (uint32_t)at << 16);
        out.resize(out.size() + ((size_t)2 << nb), 0);
        for (size_t k = 0; k < ((size_t)1 << nb); k++) put(at + k, kWalkNoEntry);
    }
    for (int i = 0; i < n; i++)
    {
        const Code &c = codes[i];
        if (c.len <= K) continue;
        const uint32_t pfx = c.code >> (c.len - K);
        const int nb = maxlen[pfx] - K, extra = c.len - K;
        const uint32_t rem = c.code & ((1u << extra) - 1u);
        const uint32_t firstk = rem << (nb - extra), cnt = 1u << (nb - extra);
        for (uint32_t k = 0; k < cnt; k++) put(sub_at[pfx] + firstk + k, single(c));
    }
    return true;
}

bool build_lut_set(const b2j_image_desc &d, std::vector<uint16_t> &out)
{
    out.assign(kLutHeader, 0);
    int built_slot[8];
    uint32_t built_off[8];
    int nbuilt = 0;
    for (int c = 0; c < 3; c++)
    {
        for (int kind = 0; kind < 2; kind++)   // 0 = DC, 1 = AC
        {
            const int th = kind == 0 ? (d.huff_id[c] >> 4) : (d.huff_id[c] & 0xF);
            if (th > 3) return false;
            const int slot = kind * 4 + th;
            if (!d.huff_present[slot]) return false;
            uint32_t off = 0;
            bool found = false;
            for (int k = 0; k < nbuilt; k++)
                if (built_slot[k] == slot) { off = built_off[k]; found = true; }
            if (!found)
            {
                std::vector<uint16_t> t;
                if (!build_huff_lut(d.huff_counts[slot], d.huff_symbols[slot], kind == 0, t, kLutMaxDecode)) return false;
                off = (uint32_t)out.size();
                out.insert(out.end(), t.begin(), t.end());
                built_slot[nbuilt] = slot; built_off[nbuilt] = off; nbuilt++;
            }
            if (off > 0xFFFF) return false;
            out[kind * 3 + c] = (uint16_t)off;
        }
    }
    while (out.size() & 7) out.push_back(0);   // 16-byte granules for the copy into shared memory
    if (out.size() > (size_t)kLutMaxDecode) return false;
    out[12] = (uint16_t)out.size();            // the decode part ends here
    // walk tables of the self-synchronising path, one per distinct table
    nbuilt = 0;
    for (int c = 0; c < 3; c++)
    {
        for (int kind = 0; kind < 2; kind++)
        {
            const int th = kind == 0 ? (d.huff_id[c] >> 4) : (d.huff_id[c] & 0xF);
            const int slot = kind * 4 + th;
            uint32_t off = 0;
            bool found = false;
            for (int k = 0; k < nbuilt; k++)
                if (built_slot[k] == slot) { off = built_off[k]; found = true; }
            if (!found)
            {
                std::vector<uint16_t> t;
                if (!build_walk_lut(d.huff_counts[slot], d.huff_symbols[slot], kind == 0, t)) return false;
                off = (uint32_t)out.size();
                out.insert(out.end(), t.begin(), t.end());
                built_slot[nbuilt] = slot; built_off[nbuilt] = off; nbuilt++;
            }
            if (off >= 0x8000) return false;   // byte offsets of the tables are kept in 16 bits
            out[6 + kind * 3 + c] = (uint16_t)off;
        }
    }
    while (out.size() & 7) out.push_back(0);
    return out.size() <= (size_t)kLutMaxEntries;
}

} // namespace b2j
