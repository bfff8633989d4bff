// Host-side checks of the encoder pieces in zstd-rs_b200/csrc/enc.cuh (the compression kernels run the same code), each against
// the decoder's own parsers in zstd-rs_b200/csrc/tables.cuh:
//   encoder_test                  unit checks; prints "ok"
//   encoder_test frame IN OUT     compresses file IN into one zstd frame (Content_Size flag set) with a simple host greedy
//                                 matcher and the block / frame writers of enc.cuh: the whole-block rehearsal that
//                                 tests/test_compress.py decodes with the oracle and with libzstd
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../zstd-rs_b200/csrc/enc.cuh"
using namespace b200z;

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)rng_state; }
#define CHECK(c, ...) do { if (!(c)) { printf(__VA_ARGS__); printf("\n"); exit(1); } } while (0)

// code lengths a HufSlot gives each symbol (entries per symbol = 2^(max_bits - len))
static void slot_lengths(const HufSlot &slot, uint32_t max_bits, uint8_t *len) {
    uint32_t cnt[256] = {0};
    for (uint32_t i = 0; i < (1u << max_bits); i++) cnt[slot.sym[i]]++;
    for (int s = 0; s < 256; s++) len[s] = cnt[s] ? (uint8_t)(max_bits - (hbs(cnt[s]) - 1)) : 0;
}

static void random_hist(uint32_t *h, uint32_t nsym, int shape) {
    memset(h, 0, 256 * 4);
    for (uint32_t i = 0; i < nsym; i++) {
        uint32_t s = nsym == 256 ? i : rnd() % 256;
        while (h[s]) s = (s + 1) % 256;
        h[s] = shape == 0 ? 1 + rnd() % 1000 : (shape == 1 ? (i == 0 ? 1000000u : 1u) : (uint32_t)(1u << (i % 24)) + rnd() % 7);
    }
}

static void test_huffman() {
    const uint32_t sizes[] = {2, 3, 5, 17, 100, 128, 129, 200, 255, 256};
    for (int it = 0; it < 3000; it++) {
        uint32_t h[256];
        const uint32_t nsym = sizes[it % 10];
        random_hist(h, nsym, it % 3);
        uint8_t len[256];
        const uint32_t mb = huf_lengths(h, len, HUF_MAX_BITS);
        uint64_t kraft = 0;
        uint32_t maxsym = 0;
        for (int s = 0; s < 256; s++) {
            CHECK(len[s] <= HUF_MAX_BITS && (len[s] > 0) == (h[s] > 0), "huf length %u for symbol %d (count %u)", len[s], s, h[s]);
            if (len[s]) { kraft += 1ull << (HUF_MAX_BITS - len[s]); maxsym = s; }
        }
        CHECK(kraft == (1ull << HUF_MAX_BITS), "kraft sum %llu, %u symbols", (unsigned long long)kraft, nsym);
        for (uint32_t form = 1; form <= 2; form++) {
            uint8_t desc[160];
            const uint32_t d = huf_write_description(desc, len, maxsym, mb, form);
            if (!d) { CHECK(form == 2 || maxsym > 128, "no direct description for %u weights", maxsym); continue; }
            uint8_t w[260];
            uint32_t nw = 0, br = 0;
            int e = huf_read_weights(desc, d, w, nw, br);
            CHECK(!e && nw == maxsym && br == d, "read_weights form %u: err %d nw %u/%u bytes %u/%u", form, e, nw, maxsym, br, d);
            HufSlot slot;
            uint32_t mb2 = 0;
            e = huf_build_table(w, nw, &slot, mb2);
            CHECK(!e && mb2 == mb, "build_table form %u: err %d max_bits %u/%u", form, e, mb2, mb);
            uint8_t len2[256];
            slot_lengths(slot, mb2, len2);
            CHECK(!memcmp(len, len2, 256), "form %u: code lengths differ after re-reading the description", form);
        }
        // one stream: encode, decode with the decoder's table
        std::vector<uint8_t> src(1 + rnd() % 3000);
        std::vector<uint8_t> present;
        for (int s = 0; s < 256; s++) if (h[s]) present.push_back((uint8_t)s);
        for (auto &b : src) b = present[rnd() % present.size()];
        uint16_t code[256];
        huf_codes(len, maxsym, mb, code);
        std::vector<uint8_t> buf(src.size() * 2 + 16, 0);
        const uint32_t n = huf_encode_stream(buf.data(), (uint32_t)buf.size(), src.data(), (uint32_t)src.size(), code, len);
        CHECK(n == huf_stream_bytes(src.data(), (uint32_t)src.size(), len), "huffman stream size");
        uint8_t wts[260];
        uint8_t desc[160];
        uint32_t nw, br, mb2;
        huf_write_description(desc, len, maxsym, mb, 0);
        huf_read_weights(desc, 160, wts, nw, br);
        HufSlot slot;
        huf_build_table(wts, nw, &slot, mb2);
        CHECK(buf[n - 1] != 0, "no end marker");
        RevBitsSmall rb{buf.data(), (int32_t)((n - 1) * 8 + hbs(buf[n - 1]) - 1)};
        for (size_t i = 0; i < src.size(); i++) {
            const int32_t p0 = rb.p;
            const uint32_t idx = rb.get(mb2);
            CHECK(slot.sym[idx] == src[i], "huffman stream symbol %zu: %u vs %u", i, slot.sym[idx], src[i]);
            rb.p = p0 - (int32_t)huf_nb(slot.nb4, idx);
        }
        CHECK(rb.p == 0, "huffman stream: %d bits left over", rb.p);
    }
}

static void test_fse() {
    for (int it = 0; it < 3000; it++) {
        const uint32_t nsym = 2 + rnd() % 52, maxlog = 5 + rnd() % 5;
        uint32_t c[64] = {0};
        uint32_t present = 0;
        for (uint32_t s = 0; s < nsym; s++) {
            if (rnd() % 4 == 0 && s + 1 != nsym) continue;
            c[s] = (it & 1) ? 1 + rnd() % 50 : (s == 0 ? 100000u : 1 + rnd() % 3);
            present++;
        }
        if (present < 2) { c[0] = 7; present += c[0] ? 0 : 1; }
        uint32_t distinct = 0, total = 0;
        for (uint32_t s = 0; s < nsym; s++) { distinct += c[s] != 0; total += c[s]; }
        const uint32_t log = fse_pick_log(total, distinct, maxlog);
        if ((1u << log) < distinct) continue;
        int16_t norm[64];
        fse_normalize(c, nsym, log, norm);
        int32_t sum = 0;
        for (uint32_t s = 0; s < nsym; s++) {
            CHECK((c[s] > 0) == (norm[s] != 0) && norm[s] >= -1, "normalized count %d for count %u", norm[s], c[s]);
            sum += norm[s] == -1 ? 1 : norm[s];
        }
        CHECK(sum == (1 << log), "normalized sum %d != %d", sum, 1 << log);
        uint8_t nc[128];
        const uint32_t nb = fse_write_ncount(nc, 128, norm, nsym, log);
        int16_t probs[256];
        uint32_t np = 0, al = 0, br = 0;
        int e = fse_read_probabilities(nc, nb, 9, 255, probs, np, al, br);
        CHECK(!e && al == log && np == nsym && br == nb, "read_probabilities: err %d log %u/%u n %u/%u bytes %u/%u", e, al, log, np, nsym, br, nb);
        for (uint32_t s = 0; s < nsym; s++) CHECK(probs[s] == norm[s], "ncount symbol %u: %d vs %d", s, probs[s], norm[s]);
        // encode a seeded string with one state, decode with the decoder's table
        FseCTab t;
        uint8_t spread[512];
        fse_build_ctab(norm, nsym, log, t, spread);
        uint32_t wide[512];
        uint16_t counter[256];
        CHECK(!fse_build_table(probs, np, al, 255, wide, counter), "build_table");
        std::vector<uint8_t> x(1 + rnd() % 2000);
        for (auto &v : x) { do v = (uint8_t)(rnd() % nsym); while (!c[v]); }
        std::vector<uint8_t> buf(x.size() * 2 + 16);
        BitW bw;
        bw.init(buf.data(), (uint32_t)buf.size());
        uint32_t st = fse_init_state(t, x.back());
        for (size_t i = x.size() - 1; i-- > 0;) fse_encode(bw, st, t, x[i]);
        fse_flush(bw, st, t);
        const uint32_t n = bw.close();
        RevBitsSmall rb{buf.data(), (int32_t)((n - 1) * 8 + hbs(buf[n - 1]) - 1)};
        uint32_t ds = rb.get(log);
        for (size_t i = 0; i < x.size(); i++) {
            CHECK((wide[ds] >> 24) == x[i], "fse symbol %zu: %u vs %u", i, wide[ds] >> 24, x[i]);
            if (i + 1 < x.size()) ds = (wide[ds] & 0xffffu) + rb.get((wide[ds] >> 16) & 0xffu);
        }
        CHECK(rb.p == 0, "fse stream: %d bits left over", rb.p);
    }
}

// ---- whole-frame rehearsal: host greedy matcher (hash of 4 bytes, one candidate per bucket, minimum match 5, inside the block)
static uint32_t ld32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static void greedy(const uint8_t *b, uint32_t n, std::vector<EncSeq> &seqs, std::vector<uint8_t> &lits) {
    std::vector<int32_t> ht(1 << 13, -1);
    uint32_t p = 0, anchor = 0;
    while (p + ENC_MIN_MATCH <= n) {
        const uint32_t h = (ld32(b + p) * 2654435761u) >> 19;
        const int32_t c = ht[h];
        ht[h] = (int32_t)p;
        uint32_t len = 0;
        if (c >= 0) while (p + len < n && b[c + len] == b[p + len]) len++;
        if (len >= ENC_MIN_MATCH) {
            seqs.push_back({p - anchor, len, p - (uint32_t)c});
            lits.insert(lits.end(), b + anchor, b + p);
            p += len; anchor = p;
        } else p++;
    }
    lits.insert(lits.end(), b + anchor, b + n);
}

static int frame(const char *in, const char *outp) {
    FILE *f = fopen(in, "rb");
    if (!f) return 2;
    std::vector<uint8_t> src;
    uint8_t tmp[65536];
    size_t r;
    while ((r = fread(tmp, 1, sizeof tmp, f)) > 0) src.insert(src.end(), tmp, tmp + r);
    fclose(f);
    std::vector<uint8_t> out(64 + src.size() + 3 * (src.size() / ENC_BLOCK + 1));
    uint32_t o = enc_frame_header(out.data(), ENC_FLAG_CONTENT_SIZE, src.size());
    const uint64_t nb = enc_num_blocks(src.size());
    std::vector<uint8_t> body(ENC_BLOCK + 64);
    static LitPlan L;
    static SeqPlan S;
    uint8_t spread[512];
    for (uint64_t b = 0; b < nb; b++) {
        const uint8_t *p = src.data() + b * ENC_BLOCK;
        const uint32_t n = (uint32_t)std::min<uint64_t>(ENC_BLOCK, src.size() - b * ENC_BLOCK);
        const uint32_t last = b + 1 == nb;
        bool same = n > 0;
        for (uint32_t i = 1; i < n && same; i++) same = p[i] == p[0];
        if (same) { enc_block_header(&out[o], last, BT_RLE, n); out[o + 3] = p[0]; o += 4; continue; }
        std::vector<EncSeq> seqs;
        std::vector<uint8_t> lits;
        if (n) greedy(p, n, seqs, lits);
        const uint32_t sz = n ? enc_block_body(lits.data(), (uint32_t)lits.size(), seqs.data(), (uint32_t)seqs.size(), body.data(), n, L, S, spread) : n;
        if (sz >= n) { enc_block_header(&out[o], last, BT_RAW, n); memcpy(&out[o + 3], p, n); o += 3 + n; }
        else { enc_block_header(&out[o], last, BT_COMPRESSED, sz); memcpy(&out[o + 3], body.data(), sz); o += 3 + sz; }
    }
    f = fopen(outp, "wb");
    if (!f) return 2;
    fwrite(out.data(), 1, o, f);
    fclose(f);
    return 0;
}

int main(int argc, char **argv) {
    if (argc == 4 && !strcmp(argv[1], "frame")) return frame(argv[2], argv[3]);
    test_huffman();
    test_fse();
    puts("ok");
    return 0;
}
