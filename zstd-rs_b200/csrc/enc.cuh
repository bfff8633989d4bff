// enc.cuh -- the serial pieces of the zstd block encoder, compiled for BOTH device and host.
//
// The compression kernels (compress.cu) call these per block or per stream; tests/host/encoder_test.cpp calls the same code on
// the host and checks every table and stream it writes against the decoder's own parsers in tables.cuh.  What they produce is
// the zstd format as ruzstd's encoder writes it (ruzstd/src/encoding/blocks/compressed.rs, huff0/huff0_encoder.rs,
// fse/fse_encoder.rs), with these choices of our own, all inside the format:
//   * Huffman code lengths are limited to 11 bits (HUF_MAX_BITS, the decoder's limit); the weights are written directly
//     (up to 128 of them) or FSE-compressed (accuracy log 6), whichever is smaller;
//   * FSE tables (LL / OF / ML, max logs 9 / 8 / 9) are normalized from the block's own histogram; a code that is the only
//     one used goes out as RLE mode.  No Predefined, Repeat or Treeless modes: every block stands alone.
//   * offsets are written as Offset_Value = offset + 3 (compressed.rs:27): no repeat-offset codes.
#pragma once
#include <stdint.h>

#include "tables.cuh"

namespace b200z {

constexpr uint32_t ENC_BLOCK = 131072;       // MAX_BLOCK_SIZE (common/mod.rs:21)
constexpr uint32_t ENC_MIN_MATCH = 5;        // the reference's minimum match
constexpr uint32_t ENC_HUF_MIN_LITERALS = 1025;   // compressed.rs:36: Huffman only for more than 1024 literals
constexpr uint32_t ENC_LL_MAX_LOG = 9, ENC_OF_MAX_LOG = 8, ENC_ML_MAX_LOG = 9;

struct EncSeq { uint32_t ll, ml, off; };   // literals before the match, match length, match offset (>= 1)

// ---- forward LSB-first bit writer (bit_io/bit_writer.rs); bytes at or past `cap` are counted, not stored
struct BitW {
    uint8_t *out;
    uint32_t pos, cap, nb;
    uint64_t acc;
    B200Z_HD void init(uint8_t *o, uint32_t c) { out = o; pos = 0; cap = c; nb = 0; acc = 0; }
    B200Z_HD void put_byte() { if (pos < cap) out[pos] = (uint8_t)acc; pos++; acc >>= 8; nb -= 8; }
    B200Z_HD void add(uint64_t v, uint32_t n) {   // n <= 32
        acc |= (v & ((1ull << n) - 1ull)) << nb;
        nb += n;
        if (nb >= 32) { put_byte(); put_byte(); put_byte(); put_byte(); }
    }
    B200Z_HD uint32_t finish() {   // pad the last byte with zeros
        while (nb >= 8) put_byte();
        if (nb) { nb = 8; put_byte(); nb = 0; }
        return pos;
    }
    B200Z_HD uint32_t close() { add(1, 1); return finish(); }   // end marker of a backward-read stream, then padding
};

// ---- sequence codes (sequence_section.rs tables; compressed.rs:245-306)
B200Z_HD uint32_t enc_ll_code(uint32_t ll, uint32_t &nbits, uint32_t &extra) {
    const uint32_t base[20] = {16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
    const uint8_t bits[20] = {1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    if (ll < 16) { nbits = 0; extra = 0; return ll; }
    int k = 19;
    while (base[k] > ll) k--;
    nbits = bits[k]; extra = ll - base[k];
    return 16 + k;
}
B200Z_HD uint32_t enc_ml_code(uint32_t ml, uint32_t &nbits, uint32_t &extra) {
    const uint32_t base[21] = {35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539};
    const uint8_t bits[21] = {1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    if (ml < 35) { nbits = 0; extra = 0; return ml - 3; }
    int k = 20;
    while (base[k] > ml) k--;
    nbits = bits[k]; extra = ml - base[k];
    return 32 + k;
}
B200Z_HD uint32_t enc_of_code(uint32_t off, uint32_t &nbits, uint32_t &extra) {
    const uint32_t v = off + 3, c = hbs(v) - 1;
    nbits = c; extra = v - (1u << c);
    return c;
}

// ---- FSE ---------------------------------------------------------------------------------------------------------
// Normalizes count[0..nsym) (total > 0, at most 1 << log present symbols) to sum 1 << log; every present symbol gets >= 1.
B200Z_HDN inline void fse_normalize(const uint32_t *count, uint32_t nsym, uint32_t log, int16_t *norm) {
    uint64_t total = 0;
    for (uint32_t s = 0; s < nsym; s++) total += count[s];
    const uint32_t size = 1u << log;
    int32_t sum = 0;
    uint32_t big = 0;
    for (uint32_t s = 0; s < nsym; s++) {
        int32_t n = 0;
        if (count[s]) {
            n = (int32_t)(((uint64_t)count[s] * size + total / 2) / total);
            if (n < 1) n = 1;
            if (count[s] > count[big]) big = s;
        }
        norm[s] = (int16_t)n;
        sum += n;
    }
    int32_t diff = (int32_t)size - sum;
    if (diff >= 0) { norm[big] = (int16_t)(norm[big] + diff); return; }
    while (diff < 0) {   // take from the largest counts, never below 1
        uint32_t m = 0;
        for (uint32_t s = 1; s < nsym; s++) if (norm[s] > norm[m]) m = s;
        int32_t take = norm[m] - 1;
        if (take > -diff) take = -diff;
        norm[m] = (int16_t)(norm[m] - take);
        diff += take;
    }
}

// Accuracy log for `n` coded symbols with `distinct` different values, at most `max_log`.
B200Z_HD uint32_t fse_pick_log(uint32_t n, uint32_t distinct, uint32_t max_log) {
    uint32_t log = hbs(n) > 2 ? hbs(n) - 2 : 1;
    if (log < 5) log = 5;
    while ((1u << log) < distinct * 2 && log < max_log) log++;
    if (log > max_log) log = max_log;
    return log;
}

// The table description read by FSETable::read_probabilities (fse_decoder.rs:224-307): nsym = last nonzero symbol + 1.
// Returns the byte count.
B200Z_HDN inline uint32_t fse_write_ncount(uint8_t *out, uint32_t cap, const int16_t *norm, uint32_t nsym, uint32_t log) {
    BitW bw;
    bw.init(out, cap);
    bw.add(log - 5, 4);
    const uint32_t sum = 1u << log;
    uint32_t counter = 0, s = 0;
    while (counter < sum && s < nsym) {
        const int32_t prob = norm[s];
        const uint32_t value = (uint32_t)(prob + 1), max_remaining = sum - counter + 1, bits = hbs(max_remaining);
        const uint32_t lt = ((1u << bits) - 1u) - max_remaining, mask = (1u << (bits - 1)) - 1u;
        if (value < lt) bw.add(value, bits - 1);
        else if (value <= mask) bw.add(value, bits);
        else bw.add(value + lt, bits);
        s++;
        if (prob != 0) counter += prob > 0 ? (uint32_t)prob : 1u;
        else {
            uint32_t z = 0;
            while (s + z < nsym && norm[s + z] == 0) z++;
            s += z;
            while (z >= 3) { bw.add(3, 2); z -= 3; }
            bw.add(z, 2);
        }
    }
    return bw.finish();
}

// Encoding table (the state-transition form of the decoder's spread, fse_decoder.rs:141-220): state values live in
// [size, 2 * size); state - size is the decoder's state index.
struct FseCTab {
    uint32_t log, rle, rle_sym, pad;
    uint16_t state[FSE_MAX_ENTRIES];
    int32_t dfs[64];     // deltaFindState
    uint32_t dnb[64];    // deltaNbBits
    uint16_t first[64];  // index in state[] of the symbol's first decoder state
};

B200Z_HDN inline void fse_build_ctab(const int16_t *norm, uint32_t nsym, uint32_t log, FseCTab &t, uint8_t *spread /* 512 */) {
    const uint32_t size = 1u << log, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
    t.log = log; t.rle = 0; t.rle_sym = 0;
    uint32_t high = size - 1;
    for (uint32_t s = 0; s < nsym; s++) if (norm[s] == -1) spread[high--] = (uint8_t)s;
    uint32_t pos = 0;
    for (uint32_t s = 0; s < nsym; s++)
        for (int32_t k = 0; k < norm[s]; k++) {
            spread[pos] = (uint8_t)s;
            pos = (pos + step) & mask;
            while (pos > high) pos = (pos + step) & mask;
        }
    uint32_t cumul[65];
    cumul[0] = 0;
    for (uint32_t s = 0; s < nsym; s++) cumul[s + 1] = cumul[s] + (norm[s] == -1 ? 1u : (uint32_t)(norm[s] > 0 ? norm[s] : 0));
    for (uint32_t s = 0; s < nsym; s++) t.first[s] = (uint16_t)cumul[s];
    for (uint32_t u = 0; u < size; u++) t.state[cumul[spread[u]]++] = (uint16_t)(size + u);
    uint32_t total = 0;
    for (uint32_t s = 0; s < nsym; s++) {
        const int32_t n = norm[s];
        if (n == 0) { t.dnb[s] = ((log + 1) << 16) - size; t.dfs[s] = 0; }
        else if (n == -1 || n == 1) { t.dnb[s] = (log << 16) - size; t.dfs[s] = (int32_t)total - 1; total++; }
        else {
            const uint32_t max_out = log - (hbs((uint32_t)n - 1) - 1), min_plus = (uint32_t)n << max_out;
            t.dnb[s] = (max_out << 16) - min_plus;
            t.dfs[s] = (int32_t)total - n;
            total += (uint32_t)n;
        }
    }
}
// first state of a stream (the last symbol encoded): the symbol's first decoder state, which always reads >= 1 bit when
// the symbol's probability is below 1 -- the Huffman-weight decoder relies on that to see the end of its stream
B200Z_HD uint32_t fse_init_state(const FseCTab &t, uint32_t s) { return t.rle ? 0u : t.state[t.first[s]]; }
B200Z_HD void fse_encode(BitW &bw, uint32_t &st, const FseCTab &t, uint32_t s) {
    if (t.rle) return;
    const uint32_t nb = (st + t.dnb[s]) >> 16;
    bw.add(st, nb);
    st = t.state[(int32_t)(st >> nb) + t.dfs[s]];
}
B200Z_HD void fse_flush(BitW &bw, uint32_t st, const FseCTab &t) { if (!t.rle) bw.add(st, t.log); }

// ---- Huffman -------------------------------------------------------------------------------------------------------
// Code lengths (<= max_len) for count[0..256) with at least 2 present symbols; Kraft sum exactly 1.  Returns the longest.
B200Z_HDN inline uint32_t huf_lengths(const uint32_t *count, uint8_t *len, uint32_t max_len) {
    uint16_t sym[256];
    uint32_t w[512];
    uint16_t parent[512];
    uint32_t n = 0;
    for (uint32_t s = 0; s < 256; s++) {
        len[s] = 0;
        if (!count[s]) continue;
        uint32_t i = n++;   // insertion sort by (count, symbol)
        while (i > 0 && count[sym[i - 1]] > count[s]) { sym[i] = sym[i - 1]; i--; }
        sym[i] = (uint16_t)s;
    }
    for (uint32_t i = 0; i < n; i++) w[i] = count[sym[i]];
    // two-queue Huffman: leaves 0..n-1 (sorted), internal nodes n..2n-2 (created in non-decreasing weight)
    uint32_t leaf = 0, node = n, next = n;
    for (uint32_t k = 0; k + 1 < n; k++) {
        uint32_t pick[2];
        for (int j = 0; j < 2; j++) {
            if (leaf < n && (node >= next || w[leaf] <= w[node])) pick[j] = leaf++;
            else pick[j] = node++;
        }
        w[next] = w[pick[0]] + w[pick[1]];
        parent[pick[0]] = parent[pick[1]] = (uint16_t)next;
        next++;
    }
    const uint32_t root = next - 1;
    uint32_t depth[512];
    depth[root] = 0;
    for (uint32_t i = root; i-- > 0;) depth[i] = depth[parent[i]] + 1;
    uint32_t maxl = 0;
    for (uint32_t i = 0; i < n; i++) {
        uint32_t d = depth[i] > max_len ? max_len : depth[i];
        len[sym[i]] = (uint8_t)d;
        if (d > maxl) maxl = d;
    }
    // Kraft repair in units of 2^-max_len
    const uint32_t T = 1u << max_len;
    uint32_t K = 0;
    for (uint32_t i = 0; i < n; i++) K += 1u << (max_len - len[sym[i]]);
    while (K > T) {   // lengthen the longest code that can still grow (least frequent first)
        uint32_t best = n, bl = 0;
        for (uint32_t i = 0; i < n; i++) { uint32_t l = len[sym[i]]; if (l < max_len && l > bl) { bl = l; best = i; } }
        K -= 1u << (max_len - bl - 1);
        len[sym[best]] = (uint8_t)(bl + 1);
    }
    while (K < T) {   // shorten the longest code whose shortening still fits (most frequent first)
        uint32_t best = n, bl = 0;
        for (uint32_t i = n; i-- > 0;) {
            uint32_t l = len[sym[i]];
            if (l > 1 && (1u << (max_len - l)) <= T - K && l > bl) { bl = l; best = i; }
        }
        K += 1u << (max_len - bl);
        len[sym[best]] = (uint8_t)(bl - 1);
    }
    maxl = 0;
    for (uint32_t i = 0; i < n; i++) if (len[sym[i]] > maxl) maxl = len[sym[i]];
    return maxl;
}

// Canonical codes in the order HuffmanTable::build_table_from_weights lays them out (huff0_decoder.rs:284-377).
B200Z_HDN inline void huf_codes(const uint8_t *len, uint32_t maxsym, uint32_t max_bits, uint16_t *code) {
    uint32_t cnt[HUF_MAX_BITS + 2] = {0}, idx[HUF_MAX_BITS + 2];
    for (uint32_t s = 0; s <= maxsym; s++) if (len[s]) cnt[len[s]]++;
    idx[max_bits] = 0;
    for (uint32_t b = max_bits; b >= 1; b--) idx[b - 1] = idx[b] + cnt[b] * (1u << (max_bits - b));
    for (uint32_t s = 0; s <= maxsym; s++) {
        const uint32_t l = len[s];
        code[s] = 0;
        if (!l) continue;
        code[s] = (uint16_t)(idx[l] >> (max_bits - l));
        idx[l] += 1u << (max_bits - l);
    }
}

// Tree description (huff0_decoder.rs:132-278 reads it): weights of symbols 0..maxsym-1, the last is implied.  Direct when
// there are at most 128 weights, FSE-compressed when that is smaller or the only option.  Returns bytes, 0 if neither fits.
// form: 0 the smaller, 1 direct only, 2 FSE only.
B200Z_HDN inline uint32_t huf_write_description(uint8_t *out, const uint8_t *len, uint32_t maxsym, uint32_t max_bits, uint32_t form = 0) {
    uint8_t wt[256];
    const uint32_t nw = maxsym;
    uint32_t hist[16] = {0};
    for (uint32_t s = 0; s < nw; s++) { wt[s] = len[s] ? (uint8_t)(max_bits + 1 - len[s]) : 0; hist[wt[s]]++; }
    const uint32_t direct = nw <= 128 && form != 2 ? 1 + (nw + 1) / 2 : 0;
    uint32_t distinct = 0;
    for (uint32_t v = 0; v < 16; v++) distinct += hist[v] != 0;
    uint32_t fse = 0;
    uint8_t tmp[160];
    if (distinct >= 2 && nw >= 2 && form != 1) {
        int16_t norm[16];
        const uint32_t log = 6;
        fse_normalize(hist, max_bits + 1, log, norm);
        uint32_t last = max_bits + 1;
        while (last > 0 && norm[last - 1] == 0) last--;
        const uint32_t hdr = fse_write_ncount(tmp + 1, 64, norm, last, log);
        FseCTab t;
        uint8_t spread[64];
        fse_build_ctab(norm, last, log, t, spread);
        BitW bw;
        bw.init(tmp + 1 + hdr, 127 - hdr);
        // decoder: state 1 decodes the even weights, state 2 the odd ones, and the stream ends when an update of the state
        // that decoded weight nw-2 runs past the start
        uint32_t st[2];
        st[(nw - 1) & 1] = fse_init_state(t, wt[nw - 1]);
        st[(nw - 2) & 1] = fse_init_state(t, wt[nw - 2]);
        for (uint32_t k = nw - 2; k-- > 0;) fse_encode(bw, st[k & 1], t, wt[k]);
        fse_flush(bw, st[1], t);
        fse_flush(bw, st[0], t);
        const uint32_t body = bw.close();
        if (hdr + body < 128) { fse = 1 + hdr + body; tmp[0] = (uint8_t)(hdr + body); }
    }
    if (direct && (!fse || direct <= fse)) {
        out[0] = (uint8_t)(127 + nw);
        for (uint32_t i = 0; i < nw; i += 2) out[1 + i / 2] = (uint8_t)((wt[i] << 4) | (i + 1 < nw ? wt[i + 1] : 0));
        return direct;
    }
    for (uint32_t i = 0; i < fse; i++) out[i] = tmp[i];
    return fse;
}

// One Huffman stream (read backward: the last symbol written is the first decoded).
B200Z_HD uint32_t huf_stream_bytes(const uint8_t *src, uint32_t n, const uint8_t *len) {
    uint32_t bits = 1;
    for (uint32_t i = 0; i < n; i++) bits += len[src[i]];
    return (bits + 7) >> 3;
}
B200Z_HDN inline uint32_t huf_encode_stream(uint8_t *out, uint32_t cap, const uint8_t *src, uint32_t n, const uint16_t *code, const uint8_t *len) {
    BitW bw;
    bw.init(out, cap);
    for (uint32_t i = n; i-- > 0;) bw.add(code[src[i]], len[src[i]]);
    return bw.close();
}
B200Z_HD void huf_stream_split(uint32_t n, uint32_t k, uint32_t &off, uint32_t &cnt) {   // 4 streams (literals_section_decoder.rs)
    const uint32_t seg = (n + 3) / 4;
    off = seg * k;
    cnt = k < 3 ? seg : n - 3 * seg;
}

// ---- literals and sequences sections ----------------------------------------------------------------------------------
struct LitPlan {
    uint32_t type, regen, hdr_size, desc_size, comp_size, max_bits, maxsym;
    uint32_t stream_size[4];
    uint8_t hdr[8];
    uint8_t desc[132];
    uint8_t len[256];
    uint16_t code[256];
};

B200Z_HD uint32_t lit_raw_header(uint8_t *h, uint32_t type, uint32_t n) {   // literals_section.rs:117-223, Raw / RLE
    if (n < 32) { h[0] = (uint8_t)(type | (n << 3)); return 1; }
    if (n < 4096) { const uint32_t v = type | (1u << 2) | (n << 4); h[0] = (uint8_t)v; h[1] = (uint8_t)(v >> 8); return 2; }
    const uint32_t v = type | (3u << 2) | (n << 4);
    h[0] = (uint8_t)v; h[1] = (uint8_t)(v >> 8); h[2] = (uint8_t)(v >> 16);
    return 3;
}

// Decides the literals type from the histogram and, for Huffman, builds the table and its description.  stream_size[] must
// then be filled (huf_stream_bytes) before lit_finish.
B200Z_HDN inline void lit_plan(const uint32_t *hist, uint32_t n, LitPlan &P) {
    P.regen = n; P.type = LT_RAW; P.desc_size = 0; P.comp_size = 0;
    uint32_t distinct = 0, maxsym = 0;
    uint64_t sumsq = 0;
    for (uint32_t s = 0; s < 256; s++) if (hist[s]) { distinct++; maxsym = s; sumsq += hist[s]; }
    P.maxsym = maxsym;
    if (n > 0 && distinct == 1) { P.type = LT_RLE; return; }
    if (n < ENC_HUF_MIN_LITERALS) return;
    P.max_bits = huf_lengths(hist, P.len, HUF_MAX_BITS);
    uint64_t bits = 0;
    for (uint32_t s = 0; s <= maxsym; s++) bits += (uint64_t)hist[s] * P.len[s];
    const uint32_t d = huf_write_description(P.desc, P.len, maxsym, P.max_bits);
    if (!d || d + 6 + bits / 8 + 4 >= n) return;   // does not pay
    huf_codes(P.len, maxsym, P.max_bits, P.code);
    P.desc_size = d;
    P.type = LT_COMPRESSED;
}
// Header and final type once the stream sizes are known; returns the section size.
B200Z_HDN inline uint32_t lit_finish(LitPlan &P) {
    if (P.type == LT_COMPRESSED) {
        P.comp_size = P.desc_size + 6 + P.stream_size[0] + P.stream_size[1] + P.stream_size[2] + P.stream_size[3];
        if (P.comp_size >= P.regen || P.stream_size[0] > 0xFFFF || P.stream_size[1] > 0xFFFF || P.stream_size[2] > 0xFFFF) P.type = LT_RAW;
    }
    if (P.type == LT_RAW) { P.hdr_size = lit_raw_header(P.hdr, LT_RAW, P.regen); return P.hdr_size + P.regen; }
    if (P.type == LT_RLE) { P.hdr_size = lit_raw_header(P.hdr, LT_RLE, P.regen); return P.hdr_size + 1; }
    const uint32_t r = P.regen, c = P.comp_size, m = r > c ? r : c;   // 4 streams: Size_Format 1..3
    if (m < 1024) {
        const uint32_t v = LT_COMPRESSED | (1u << 2) | (r << 4) | (c << 14);
        for (int i = 0; i < 3; i++) P.hdr[i] = (uint8_t)(v >> (8 * i));
        P.hdr_size = 3;
    } else if (m < 16384) {
        const uint32_t v = LT_COMPRESSED | (2u << 2) | (r << 4) | (c << 18);
        for (int i = 0; i < 4; i++) P.hdr[i] = (uint8_t)(v >> (8 * i));
        P.hdr_size = 4;
    } else {
        const uint64_t v = LT_COMPRESSED | (3u << 2) | ((uint64_t)r << 4) | ((uint64_t)c << 22);
        for (int i = 0; i < 5; i++) P.hdr[i] = (uint8_t)(v >> (8 * i));
        P.hdr_size = 5;
    }
    return P.hdr_size + P.comp_size;
}

struct SeqPlan {
    uint32_t nseq, hdr_size;
    uint8_t hdr[4 + 192];   // Number_of_Sequences, Symbol_Compression_Modes, then the LL / OF / ML descriptions
    FseCTab ll, of, ml;
};

// hll[36], hof[32], hml[53]: histograms of the codes.  `spread` = 512 bytes of scratch.
B200Z_HDN inline void seq_plan(uint32_t nseq, const uint32_t *hll, const uint32_t *hof, const uint32_t *hml, SeqPlan &P, uint8_t *spread) {
    P.nseq = nseq;
    uint32_t h = 0;
    if (nseq < 128) P.hdr[h++] = (uint8_t)nseq;
    else if (nseq < 0x7F00) { P.hdr[h++] = (uint8_t)((nseq >> 8) + 0x80); P.hdr[h++] = (uint8_t)nseq; }
    else { P.hdr[h++] = 0xFF; P.hdr[h++] = (uint8_t)(nseq - 0x7F00); P.hdr[h++] = (uint8_t)((nseq - 0x7F00) >> 8); }
    if (nseq == 0) { P.hdr_size = h; return; }
    const uint32_t modes_at = h++;
    uint32_t modes = 0;
    const uint32_t *hists[3] = {hll, hof, hml};
    const uint32_t nsyms[3] = {36, 32, 53}, maxlogs[3] = {ENC_LL_MAX_LOG, ENC_OF_MAX_LOG, ENC_ML_MAX_LOG}, shifts[3] = {6, 4, 2};
    FseCTab *tabs[3] = {&P.ll, &P.of, &P.ml};
    for (int k = 0; k < 3; k++) {
        const uint32_t *c = hists[k];
        uint32_t distinct = 0, last = 0;
        for (uint32_t s = 0; s < nsyms[k]; s++) if (c[s]) { distinct++; last = s; }
        FseCTab &t = *tabs[k];
        if (distinct == 1) {
            t.rle = 1; t.rle_sym = last; t.log = 0;
            modes |= MODE_RLE << shifts[k];
            P.hdr[h++] = (uint8_t)last;
            continue;
        }
        const uint32_t log = fse_pick_log(nseq, distinct, maxlogs[k]);
        int16_t norm[64];
        fse_normalize(c, last + 1, log, norm);
        h += fse_write_ncount(P.hdr + h, 96, norm, last + 1, log);
        fse_build_ctab(norm, last + 1, log, t, spread);
        modes |= MODE_FSE << shifts[k];
    }
    P.hdr[modes_at] = (uint8_t)modes;
    P.hdr_size = h;
}

// The sequences bitstream (sequence_section_decoder.rs reads it from the end): last sequence first.
B200Z_HDN inline uint32_t seq_encode(uint8_t *out, uint32_t cap, const EncSeq *seqs, uint32_t n, const SeqPlan &P) {
    BitW bw;
    bw.init(out, cap);
    uint32_t llb, lle, mlb, mle, ofb, ofe;
    const EncSeq &z = seqs[n - 1];
    uint32_t sll = fse_init_state(P.ll, enc_ll_code(z.ll, llb, lle));
    uint32_t sof = fse_init_state(P.of, enc_of_code(z.off, ofb, ofe));
    uint32_t sml = fse_init_state(P.ml, enc_ml_code(z.ml, mlb, mle));
    bw.add(lle, llb); bw.add(mle, mlb); bw.add(ofe, ofb);
    for (uint32_t i = n - 1; i-- > 0;) {
        const EncSeq &q = seqs[i];
        const uint32_t lc = enc_ll_code(q.ll, llb, lle), mc = enc_ml_code(q.ml, mlb, mle), oc = enc_of_code(q.off, ofb, ofe);
        fse_encode(bw, sof, P.of, oc);
        fse_encode(bw, sml, P.ml, mc);
        fse_encode(bw, sll, P.ll, lc);
        bw.add(lle, llb); bw.add(mle, mlb); bw.add(ofe, ofb);
    }
    fse_flush(bw, sml, P.ml);
    fse_flush(bw, sof, P.of);
    fse_flush(bw, sll, P.ll);
    return bw.close();
}

// ---- block body: [literals section][sequences section] (block_decoder.rs:97-197 reads it) ----------------------------------
// The pieces, in the order the kernels run them (k_cblock spreads the streams over lanes); enc_block_body runs them serially.
B200Z_HD void enc_histograms(const uint8_t *lits, uint32_t nlit, const EncSeq *seqs, uint32_t nseq, uint32_t *hist, uint32_t *hll, uint32_t *hof,
                             uint32_t *hml, uint32_t lane, uint32_t nlanes) {   // counts only add up: callers zero and combine
    uint32_t b, e;
    for (uint32_t i = lane; i < nlit; i += nlanes) hist[lits[i]]++;
    for (uint32_t i = lane; i < nseq; i += nlanes) { hll[enc_ll_code(seqs[i].ll, b, e)]++; hof[enc_of_code(seqs[i].off, b, e)]++; hml[enc_ml_code(seqs[i].ml, b, e)]++; }
}
// Writes everything of the literals section except the Huffman streams; returns the offset of stream 0 (or the section end).
B200Z_HDN inline uint32_t lit_write_prefix(uint8_t *out, const LitPlan &L, const uint8_t *lits) {
    uint32_t p = 0;
    for (uint32_t i = 0; i < L.hdr_size; i++) out[p++] = L.hdr[i];
    if (L.type == LT_RAW) { for (uint32_t i = 0; i < L.regen; i++) out[p++] = lits[i]; return p; }
    if (L.type == LT_RLE) { out[p++] = lits[0]; return p; }
    for (uint32_t i = 0; i < L.desc_size; i++) out[p++] = L.desc[i];
    for (int k = 0; k < 3; k++) { out[p++] = (uint8_t)L.stream_size[k]; out[p++] = (uint8_t)(L.stream_size[k] >> 8); }
    return p;
}
// Writes the sequences section at `out` (room `cap`); returns its size (> cap: did not fit, nothing beyond cap written).
B200Z_HDN inline uint32_t seq_write(uint8_t *out, uint32_t cap, const EncSeq *seqs, const SeqPlan &S) {
    if (S.hdr_size > cap) return cap + 1;
    for (uint32_t i = 0; i < S.hdr_size; i++) out[i] = S.hdr[i];
    if (!S.nseq) return S.hdr_size;
    return S.hdr_size + seq_encode(out + S.hdr_size, cap - S.hdr_size, seqs, S.nseq, S);
}
B200Z_HDN inline uint32_t enc_block_body(const uint8_t *lits, uint32_t nlit, const EncSeq *seqs, uint32_t nseq, uint8_t *out, uint32_t cap, LitPlan &L,
                                         SeqPlan &S, uint8_t *spread) {
    uint32_t hist[256] = {0}, hll[36] = {0}, hof[32] = {0}, hml[53] = {0};
    enc_histograms(lits, nlit, seqs, nseq, hist, hll, hof, hml, 0, 1);
    lit_plan(hist, nlit, L);
    if (L.type == LT_COMPRESSED)
        for (uint32_t k = 0; k < 4; k++) { uint32_t o, c; huf_stream_split(nlit, k, o, c); L.stream_size[k] = huf_stream_bytes(lits + o, c, L.len); }
    const uint32_t lsz = lit_finish(L);
    if (lsz > cap) return cap + 1;
    uint32_t p = lit_write_prefix(out, L, lits);
    if (L.type == LT_COMPRESSED)
        for (uint32_t k = 0; k < 4; k++) { uint32_t o, c; huf_stream_split(nlit, k, o, c); p += huf_encode_stream(out + p, L.stream_size[k], lits + o, c, L.code, L.len); }
    seq_plan(nseq, hll, hof, hml, S, spread);
    return lsz + seq_write(out + lsz, cap - lsz, seqs, S);
}

// ---- frame and block headers (encoding/frame_header.rs, block_header.rs) -------------------------------------------------
constexpr uint32_t ENC_FLAG_CHECKSUM = 1u, ENC_FLAG_CONTENT_SIZE = 2u;

// Frame_Content_Size field bytes written for `n` (the 1-byte field needs Single_Segment, which these frames never set)
B200Z_HD uint32_t enc_fcs_bytes(uint64_t n) { return n < 256 ? 4u : (n < 65536 ? 2u : (n >> 32 ? 8u : 4u)); }
B200Z_HD uint32_t enc_frame_header(uint8_t *h, uint32_t flags, uint64_t n) {
    const uint32_t fb = (flags & ENC_FLAG_CONTENT_SIZE) ? enc_fcs_bytes(n) : 0;
    const uint32_t fcs_flag = fb == 2 ? 1u : (fb == 4 ? 2u : (fb == 8 ? 3u : 0u));
    h[0] = 0x28; h[1] = 0xB5; h[2] = 0x2F; h[3] = 0xFD;
    h[4] = (uint8_t)((fcs_flag << 6) | ((flags & ENC_FLAG_CHECKSUM) ? 4u : 0u));
    h[5] = (uint8_t)((17 - 10) << 3);   // Window_Descriptor: 128 KiB
    const uint64_t v = fb == 2 ? n - 256 : n;
    for (uint32_t i = 0; i < fb; i++) h[6 + i] = (uint8_t)(v >> (8 * i));
    return 6 + fb;
}
B200Z_HD void enc_block_header(uint8_t *h, uint32_t last, uint32_t type, uint32_t size) {
    const uint32_t v = (size << 3) | (type << 1) | last;
    h[0] = (uint8_t)v; h[1] = (uint8_t)(v >> 8); h[2] = (uint8_t)(v >> 16);
}
// blocks of an n-byte frame: the reference fills 128 KiB blocks until a read returns nothing, so a multiple of 128 KiB
// (and the empty input) ends with an empty Raw block (frame_compressor.rs:141-186)
B200Z_HD uint64_t enc_num_blocks(uint64_t n) { return n / ENC_BLOCK + 1; }

}  // namespace b200z
