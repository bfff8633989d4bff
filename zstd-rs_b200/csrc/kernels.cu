// kernels.cu -- sm_100a kernels of the zstd block-decompression hot path.
//
//   k_predefined : the three predefined FSE LUTs, built once per context
//   k_setup      : per block: Huffman tree description -> huff0 LUT, FSE table descriptions -> LL/OF/ML LUTs
//                  (HuffmanTable::build_decoder huff0_decoder.rs:117, maybe_update_fse_tables
//                  sequence_section_decoder.rs:294-410)
//   k_huf        : literals: one lane per huff0 stream (decompress_literals literals_section_decoder.rs:40-158)
//   k_fse        : sequences: one lane per block walks the reversed bitstream with three interleaved FSE states
//                  (decode_sequences sequence_section_decoder.rs:14-221)
//   k_exec       : LZ77 execution into the frame's output (execute_sequences sequence_execution.rs:5-118,
//                  DecodeBuffer::{push,repeat,repeat_from_dict} decode_buffer.rs:74-179), one warp per frame,
//                  blocks of a frame in order
//
// Integer/byte work only; the roofline is HBM bandwidth (DESIGN.md section 4).
#include <cuda_runtime.h>
#include <limits.h>
#include <stdlib.h>
#include <stdint.h>

#include "kernels.h"
#include "setup.cuh"
#include "xxh64.cuh"

namespace b200z {

// ------------------------------------------------------------------------------------------------------------
__global__ void k_predefined(FseSlot *predef) {
    uint32_t k = threadIdx.x;
    if (k < 3) fse_build_predefined(k, k == 0 ? &predef->ll : (k == 1 ? &predef->of : &predef->ml));
}

// ------------------------------------------------------------------------------------------------------------
// k_setup: one WARP per block.  Lane 0 walks the bit-serial descriptions; the table expansion is warp-parallel
// out of shared memory (setup.cuh).  Tables land in global slots (3 KiB huff0 / 3 x 1 KiB FSE) that the decode
// kernels stage into shared memory.
// ------------------------------------------------------------------------------------------------------------
constexpr int SETUP_WARPS = 4;

__device__ int setup_seq_table_warp(SetupScratch &sc, uint32_t mode, const uint8_t *&p, uint32_t &rem, uint32_t max_log, uint32_t max_sym,
                                    FseTab *tab, int missing_err) {
    const uint32_t lane = lane_id();
    if (mode == MODE_FSE) {
        uint32_t used = 0, nprobs = 0, log = 0;
        int e = 0;
        if (lane == 0) e = fse_read_probabilities(p, rem, max_log, max_sym, sc.probs, nprobs, log, used);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e) return e;
        used = __shfl_sync(0xffffffffu, used, 0); nprobs = __shfl_sync(0xffffffffu, nprobs, 0); log = __shfl_sync(0xffffffffu, log, 0);
        __syncwarp();
        e = fse_build_warp(sc, nprobs, log, max_sym, tab);
        if (e) return e;
        p += used; rem -= used;
    } else if (mode == MODE_RLE) {
        if (rem == 0) return missing_err;
        uint32_t sym = p[0];
        if (sym > max_sym) return B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_ML_TABLE;  // sic, sequence_section_decoder.rs:321,356,391
        if (lane == 0) { tab->log = 0; tab->valid = 1; tab->is_rle = 1; tab->e[0] = fse_pack16(0, 0, 0, sym); }
        p += 1; rem -= 1;
    }
    return 0;
}

__global__ void __launch_bounds__(SETUP_WARPS * 32) k_setup(const BlockDesc *__restrict__ descs, BlockAux *__restrict__ aux,
                                                          const uint8_t *__restrict__ input, uint32_t nblocks, uint32_t parts) {
    // parts: bit 0 = the literals side (Huffman table + its BlockAux fields), bit 1 = the sequences side (FSE tables + the rest of
    // BlockAux).  The two sides are independent: the shipped launch order runs them as two launches on two streams.
    __shared__ SetupScratch scratch[SETUP_WARPS];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t b = blockIdx.x * SETUP_WARPS + warp;
    if (b >= nblocks) return;
    SetupScratch &sc = scratch[warp];
    const BlockDesc &d = descs[b];
    uint32_t st_lit = 0, st_seq = 0, lit_streams_off = 0, seq_bits_off = 0;
    if (d.btype == BT_COMPRESSED && !(d.host_status && (d.host_status >> 24) == 1)) {
        const uint8_t *content = input + d.src_off;
        if (!(parts & 1u)) {
        } else if (d.lit_type == LT_COMPRESSED) {
            uint32_t used = 0, nweights = 0;
            int e = 0;
            if (lane == 0) e = huf_read_weights_scratch(content + d.lit_off, d.lit_comp_size, sc.weights, nweights, used, sc.probs, sc.wtab, sc.wcount);
            e = __shfl_sync(0xffffffffu, e, 0);
            used = __shfl_sync(0xffffffffu, used, 0); nweights = __shfl_sync(0xffffffffu, nweights, 0);
            __syncwarp();
            if (!e) e = huf_build_warp(sc, nweights, d.huf_build);
            if (e) { st_lit = mk_status((uint32_t)e, B200Z_STAGE_LITERALS); if (lane == 0) { d.huf_build->max_bits = 0; d.huf_build->status = (uint32_t)e; } }
            lit_streams_off = used;
        } else if (d.lit_type == LT_TREELESS) {
            if (d.huf == nullptr) st_lit = mk_status(B200Z_ERR_LIT_UNINITIALIZED_HUFFMAN_TABLE, B200Z_STAGE_LITERALS);
        }
        if ((parts & 2u) && d.nseq != 0 && !d.host_status) {
            // a table whose build fails (or is never reached) must read as uninitialised to every later user of the slot
            if (lane == 0 && d.fse_build) { d.fse_build->ll.valid = 0; d.fse_build->ll.log = 0; d.fse_build->of.valid = 0; d.fse_build->of.log = 0; d.fse_build->ml.valid = 0; d.fse_build->ml.log = 0; }
            __syncwarp();
            const uint8_t *p = content + d.seq_off;
            uint32_t rem = d.src_size - d.seq_off;
            int e = setup_seq_table_warp(sc, d.modes >> 6, p, rem, 9, 35, d.fse_build ? &d.fse_build->ll : nullptr, B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_LL_TABLE);
            __syncwarp();
            if (!e) e = setup_seq_table_warp(sc, (d.modes >> 4) & 3, p, rem, 8, 31, d.fse_build ? &d.fse_build->of : nullptr, B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_OF_TABLE);
            __syncwarp();
            if (!e) e = setup_seq_table_warp(sc, (d.modes >> 2) & 3, p, rem, 9, 52, d.fse_build ? &d.fse_build->ml : nullptr, B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_ML_TABLE);
            if (e) st_seq = mk_status((uint32_t)e, B200Z_STAGE_SEQUENCES);
            seq_bits_off = (uint32_t)(p - content);
        }
    }
    if (lane == 0) {
        BlockAux &a = aux[b];
        if (parts & 1u) { a.status = st_lit; a.lit_streams_off = lit_streams_off; }   // literals-stage status; the sequence-stage status travels in `pad` until k_exec orders them
        if (parts & 2u) {
            a.out_size = 0; a.seq_bits_off = seq_bits_off; a.sum_ll = 0; a.pad = st_seq;
            a.hist_after[0] = a.hist_after[1] = a.hist_after[2] = 0; a.flags = 0; a.ready = 0; a.progress = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// k_huf: literals.  One CTA (one warp) = 8 blocks x 4 streams; the 8 huff0 LUTs (3 KiB each, split symbol /
// 4-bit length) are staged into shared memory; every lane walks its own reversed bitstream -- one 64-bit window
// (PosRing: 3 LDS + 2 funnel shifts) per four symbols -- and writes its symbols in 16-byte vectors.
// ------------------------------------------------------------------------------------------------------------
constexpr uint32_t HUF_BLOCKS_PER_CTA = 8;
constexpr uint32_t HUF_SMEM_PER_BLOCK = HUF_TABLE_ENTRIES + HUF_TABLE_ENTRIES / 2;  // 3072

// ---- PTX helpers with defined behaviour for shift counts >= 32 (shl/shr clamp the count, funnelshift .clamp)
__device__ __forceinline__ uint32_t shr_c(uint32_t a, uint32_t n) { uint32_t r; asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(n)); return r; }
__device__ __forceinline__ uint32_t shl_c(uint32_t a, uint32_t n) { uint32_t r; asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(n)); return r; }
__device__ __forceinline__ uint32_t fsl_c(uint32_t lo, uint32_t hi, uint32_t n) { return __funnelshift_lc(lo, hi, n); }
__device__ __forceinline__ uint32_t bfind32(uint32_t a) { uint32_t r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(a)); return r; }   // floor(log2 a)

constexpr uint32_t RING_STRIDE = 144;   // bytes of shared memory per bitstream: a mirror group + 8 groups of 16 bytes (PosRing)

// ---- shared-memory accessors by 32-bit shared address
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint2 lds64(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint4 lds128(uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) { asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ void red_or_shared(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }


// Position-based reversed bit reader for the fast paths of k_fse and k_huf.  The only state is P = bits_remaining()
// (bit_reader_reverse.rs:27-29); every read assembles the 64 bits below position P from three words of a per-lane
// shared-memory ring (8 groups of 16 bytes + a mirror of the top group below slot 0, so that the three words are
// always at a0, a0 - 4, a0 - 8) that cp.async keeps filled 7 groups ahead of consumption.  No window registers,
// no refill / skip bookkeeping: a step costs 3 LDS + 2 funnel shifts.  Bits below the stream start are NOT
// zeroed here: reading them makes P negative, which the caller checks (the block is then replayed by the exact
// path, whose reader zero-fills like BitReaderReversed, bit_reader_reverse.rs:57-83).
struct PosRing {
    const uint4 *base;   // 16-byte aligned address at or below the stream start
    uint32_t ring;       // shared-memory byte address of slot 0 (the mirror slot is at ring - 16)
    int32_t gm1;         // bit offset of the stream's first byte inside group 0, minus 1
    int32_t next_g;      // next group to request (descending)
    int32_t P;           // bits_remaining()

    __device__ __forceinline__ uint32_t lds(uint32_t addr) const { uint32_t w; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(addr) : "memory"); return w; }
    // request group g when `on` (predicated, no branch): slot g & 7, plus the mirror below slot 0 for slot 7
    __device__ __forceinline__ void request(int32_t g, bool on) {
        const uint32_t slot = (uint32_t)g & 7u;
        const uint32_t dst = ring + (slot << 4);
        const uint4 *src = base + g;
        const uint32_t p1 = on ? 1u : 0u, p2 = (on && slot == 7u) ? 1u : 0u;
        asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %3, 0;\n\tsetp.ne.u32 q, %4, 0;\n\t"
                     "@p cp.async.cg.shared.global [%0], [%2], 16;\n\t@q cp.async.cg.shared.global [%1], [%2], 16;\n\t"
                     "cp.async.commit_group;\n\t}" ::"r"(dst), "r"(ring - 16u), "l"(src), "r"(p1), "r"(p2) : "memory");
    }
    __device__ __forceinline__ bool init(const uint8_t *src, uint32_t len, uint32_t ring_slot0) {
        ring = ring_slot0; base = nullptr; gm1 = -1; next_g = -1; P = 0;
        if (len == 0) return false;
        const uint32_t last = src[len - 1];
        if (last == 0) return false;
        const uintptr_t a = (uintptr_t)src;
        base = (const uint4 *)(a & ~(uintptr_t)15);
        gm1 = (int32_t)((uint32_t)(a & 15) * 8u) - 1;
        P = (int32_t)((len - 1) * 8u + (31u - (uint32_t)__clz((int)last)));
        const int32_t gt = (gm1 + P) >> 7;    // group of the first data bit (-1 only for an empty stream at offset 0)
        for (int32_t g = gt; g > gt - 8; g--) request(g, g >= 0);
        next_g = gt - 8;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        return true;
    }
    // the 64 bits below position P, left aligned in hi:lo (garbage once P < 64 bits from the stream start: unused)
    __device__ __forceinline__ void window(uint32_t &hi, uint32_t &lo) const {
        const int32_t G = gm1 + P;                               // bit index (from `base`) of the next unread bit
        const uint32_t a0 = ring + (((uint32_t)G >> 3) & 0x7cu);  // word (G >> 5) & 31 of the ring
        const uint32_t A = lds(a0), B = lds(a0 - 4u), C = lds(a0 - 8u);
        const uint32_t sh = ~(uint32_t)G;                         // 31 - (G & 31), the funnel shift uses the low 5 bits
        hi = __funnelshift_l(B, A, sh);
        lo = __funnelshift_l(C, B, sh);
    }
    // Keeps the ring 7 groups ahead.  Call at least once per 116 consumed bits (every second sequence): consumption
    // then leaves at most one group per call, so one request per call keeps up; the groups a step can touch before
    // the next call (down to 2 below the current one) are complete after wait_group 5.
    __device__ __forceinline__ void service() {
        const int32_t gh = (gm1 + P) >> 7;
        const bool need = next_g >= gh - 7;
        request(next_g, need && next_g >= 0);
        next_g -= need ? 1 : 0;
        asm volatile("cp.async.wait_group 5;" ::: "memory");
    }
};

// Reversed bit reader for the decode kernels: 64-bit window hi:lo (left aligned) fed by ALIGNED 128-bit loads,
// double buffered (`nxt` is requested a whole 16-byte group before it is needed, so L2/HBM latency overlaps
// ~25-50 symbols of decoding).  Same observable behaviour as BitReaderReversed (bit_reader_reverse.rs:6-162):
// bits below the stream start read as zero and `p` = bits_remaining() goes negative.
struct HufBits {
    const uint4 *base;  // 16-byte aligned address at or below the stream start
    uint4 cur, nxt;     // word groups curg and curg - 1
    uint32_t hi, lo;    // unread bits, left aligned in hi:lo
    int32_t fill;       // bits in hi:lo (virtual zeros below the stream start count)
    int32_t wi;         // 32-bit words [0, wi) not consumed yet
    int32_t curg;
    int32_t sw;         // index of the word holding the stream's first byte
    uint32_t smask;     // mask of the bits of word `sw` that belong to the stream
    int32_t p;          // bits_remaining()
    __device__ __forceinline__ uint4 group(int32_t g) const { return g >= 0 ? __ldg(base + g) : make_uint4(0, 0, 0, 0); }
    __device__ __forceinline__ uint32_t next_word() {
        int32_t i = wi - 1;
        uint32_t w = 0;
        if (i >= 0) {
            int32_t g = i >> 2;
            if (g != curg) { cur = nxt; curg = g; nxt = group(g - 1); }
            uint32_t k = (uint32_t)i & 3u;
            w = k == 0 ? cur.x : (k == 1 ? cur.y : (k == 2 ? cur.z : cur.w));
            if (i < sw) w = 0; else if (i == sw) w &= smask;
            wi = i;
        }
        return w;
    }
    __device__ __forceinline__ bool init(const uint8_t *src, uint32_t len) {
        if (len == 0) return false;
        uint32_t last = src[len - 1];
        if (last == 0) return false;
        uintptr_t a = (uintptr_t)src;
        base = (const uint4 *)(a & ~(uintptr_t)15);
        uint32_t g0 = (uint32_t)(a & 15) * 8u;
        sw = (int32_t)(g0 >> 5);
        smask = ~((1u << (g0 & 31u)) - 1u);
        p = (int32_t)((len - 1) * 8u + (31u - (uint32_t)__clz((int)last)));
        hi = lo = 0; fill = 0; wi = 0; curg = -1;
        cur = nxt = make_uint4(0, 0, 0, 0);
        if (p > 0) {
            uint32_t gtop = g0 + (uint32_t)p - 1u;
            wi = (int32_t)(gtop >> 5) + 1;
            curg = (wi - 1) >> 2;
            cur = group(curg); nxt = group(curg - 1);
            uint32_t w = next_word();
            uint32_t used = (gtop & 31u) + 1u;
            hi = w << (32u - used);
            fill = (int32_t)used;
        }
        return true;
    }
    // afterwards fill > 32: at least 32 real-or-virtual bits ready
    __device__ __forceinline__ void refill() {
        if (fill <= 32) {
            uint32_t w = next_word();
            if (fill == 32) lo = w;
            else if (fill == 0) hi = w;
            else { hi |= w >> fill; lo = w << (32 - fill); }   // fill in [1, 31]
            fill += 32;
        }
    }
    __device__ __forceinline__ void skip(uint32_t n) {  // n <= 31
        hi = __funnelshift_l(lo, hi, n);
        lo <<= n;
        fill -= (int32_t)n;
        p -= (int32_t)n;
    }
};

// Fast huff0 stream: decodes exactly `cap` symbols with a count-based, branch-free loop (no per-symbol position
// checks); the stream was "regular" iff it is then exhausted exactly (every code consumes >= 1 bit, so ending on
// bits_remaining == 0 after `cap` symbols is equivalent to the reference's loop stopping there,
// literals_section_decoder.rs:112-121).  Returns true when regular; otherwise the caller replays with huf_stream2.
__device__ __forceinline__ bool huf_stream_fast(const uint8_t *__restrict__ tsym, const uint8_t *__restrict__ tnb, uint32_t mb,
                                                const uint8_t *src, uint32_t len, uint8_t *dst, uint32_t cap, uint32_t ring_addr) {
    PosRing br;
    if (!br.init(src, len, ring_addr + 16u)) return false;   // slot 0 of the ring; the mirror slot sits below it
    const uint32_t sh = 32u - mb;
    uint32_t a_sym = (uint32_t)__cvta_generic_to_shared(tsym), a_nb = (uint32_t)__cvta_generic_to_shared(tnb);
    asm volatile("" : "+r"(a_sym), "+r"(a_nb));
    // one symbol out of the window hi:lo (left aligned): LUT index = the top max_bits bits (huff0_decoder.rs:25-53)
    auto sym1 = [&](uint32_t &hi, uint32_t &lo, uint32_t &used) -> uint32_t {
        const uint32_t idx = hi >> sh;
        const uint32_t s = lds8(a_sym + idx);
        const uint32_t nb = (lds8(a_nb + (idx >> 1)) >> ((idx & 1u) * 4u)) & 15u;
        hi = __funnelshift_l(lo, hi, nb);
        lo <<= nb;
        used += nb;
        return s;
    };
    auto one = [&]() -> uint32_t { uint32_t hi, lo, used = 0; br.window(hi, lo); const uint32_t s = sym1(hi, lo, used); br.P -= (int32_t)used; br.service(); return s; };
    uint32_t n = 0;
    // scalar head until dst + n is 16-byte aligned
    uint32_t head = (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u);
    if (head > cap) head = cap;
    for (; n < head; n++) dst[n] = (uint8_t)one();
    // 16 symbols per store; a window of 64 bits feeds four symbols (<= 44 bits)
    for (; n + 16 <= cap; n += 16) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t hi, lo, used = 0;
            br.window(hi, lo);
            const uint32_t s0 = sym1(hi, lo, used), s1 = sym1(hi, lo, used), s2 = sym1(hi, lo, used), s3 = sym1(hi, lo, used);
            br.P -= (int32_t)used;
            if (q & 1) br.service();                  // every 8 symbols (<= 88 bits)
            w[q] = s0 | (s1 << 8) | (s2 << 16) | (s3 << 24);
        }
        *reinterpret_cast<uint4 *>(dst + n) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    for (; n < cap; n++) dst[n] = (uint8_t)one();
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    return br.P == 0;
}

// returns 0 exhausted exactly, 1 over-read, 2 cap reached, 3 ExtraPadding
__device__ __forceinline__ int huf_stream2(const uint8_t *__restrict__ tsym, const uint8_t *__restrict__ tnb, uint32_t mb,
                                           const uint8_t *src, uint32_t len, uint8_t *dst, uint32_t store_limit, uint32_t cap, uint32_t &count) {
    HufBits br;
    count = 0;
    if (!br.init(src, len)) return 3;
    uint32_t n = 0;
    const uint32_t sh = 32u - mb;
    // scalar head until dst + n is 16-byte aligned
    while (br.p > 0 && n < cap && (((uintptr_t)(dst + n)) & 15u)) {
        br.refill();
        uint32_t idx = br.hi >> sh;
        if (n < store_limit) dst[n] = tsym[idx];
        n++;
        br.skip((tnb[idx >> 1] >> ((idx & 1u) * 4u)) & 15u);
    }
    // vector body: 16 symbols per store while at least 16 full-length codes remain
    while (br.p >= (int32_t)(16 * HUF_MAX_BITS) && n + 16 <= cap && n + 16 <= store_limit) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t acc = 0;
#pragma unroll
            for (int k = 0; k < 4; k += 2) {
                br.refill();   // > 32 bits: two codes of <= 11 bits
                uint32_t i0 = br.hi >> sh;
                uint32_t s0 = tsym[i0];
                br.skip((tnb[i0 >> 1] >> ((i0 & 1u) * 4u)) & 15u);
                uint32_t i1 = br.hi >> sh;
                uint32_t s1 = tsym[i1];
                br.skip((tnb[i1 >> 1] >> ((i1 & 1u) * 4u)) & 15u);
                acc |= (s0 << (8 * k)) | (s1 << (8 * k + 8));
            }
            w[q] = acc;
        }
        *reinterpret_cast<uint4 *>(dst + n) = make_uint4(w[0], w[1], w[2], w[3]);
        n += 16;
    }
    // scalar tail
    while (br.p > 0) {
        if (n == cap) { count = n; return 2; }
        br.refill();
        uint32_t idx = br.hi >> sh;
        if (n < store_limit) dst[n] = tsym[idx];
        n++;
        br.skip((tnb[idx >> 1] >> ((idx & 1u) * 4u)) & 15u);
    }
    count = n;
    return br.p == 0 ? 0 : 1;
}

__global__ void __launch_bounds__(32) k_huf(const BlockDesc *__restrict__ descs, BlockAux *__restrict__ aux, const uint8_t *__restrict__ input,
                                          uint8_t *__restrict__ lit_scratch, uint32_t nblocks) {
    extern __shared__ __align__(16) uint8_t smem_huf[];
    const uint32_t lane = threadIdx.x;
    const uint32_t b0 = blockIdx.x * HUF_BLOCKS_PER_CTA;
    const uint32_t g = lane >> 2, k = lane & 3;
    const uint32_t b = b0 + g;
    bool active = b < nblocks;
    const BlockDesc *d = nullptr;
    bool work = false;
    uint32_t err = 0;
    const HufSlot *slot = nullptr;
    if (active) {
        d = &descs[b];
        work = d->btype == BT_COMPRESSED && (d->lit_type == LT_COMPRESSED || d->lit_type == LT_TREELESS) &&
               !(d->host_status && (d->host_status >> 24) == 1) && aux[b].status == 0;
        if (work) {
            slot = d->huf;
            if (slot == nullptr || slot->max_bits == 0) { err = B200Z_ERR_LIT_UNINITIALIZED_HUFFMAN_TABLE; work = false; }
        }
    }
    // ---- stage the LUTs: group j's table is copied by the whole warp, 16 bytes per lane per step
    for (uint32_t j = 0; j < HUF_BLOCKS_PER_CTA; j++) {
        unsigned long long sp = __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)(work ? slot : nullptr), j * 4);
        if (!sp) continue;
        const HufSlot *s = (const HufSlot *)(uintptr_t)sp;
        uint32_t mbj = s->max_bits;
        uint32_t n_sym16 = ((1u << mbj) + 15) >> 4, n_nb16 = (((1u << mbj) >> 1) + 15) >> 4;
        uint4 *dsym = reinterpret_cast<uint4 *>(smem_huf + j * HUF_SMEM_PER_BLOCK);
        uint4 *dnb = reinterpret_cast<uint4 *>(smem_huf + j * HUF_SMEM_PER_BLOCK + HUF_TABLE_ENTRIES);
        const uint4 *ssym = reinterpret_cast<const uint4 *>(s->sym);
        const uint4 *snb = reinterpret_cast<const uint4 *>(s->nb4);
        for (uint32_t i = lane; i < n_sym16; i += 32) dsym[i] = ssym[i];
        for (uint32_t i = lane; i < n_nb16; i += 32) dnb[i] = snb[i];
    }
    __syncwarp();
    const uint8_t *tsym = smem_huf + g * HUF_SMEM_PER_BLOCK;
    const uint8_t *tnb = tsym + HUF_TABLE_ENTRIES;

    int rc = 0; uint32_t count = 0; bool irregular = false;
    if (work) {
        uint32_t so = aux[b].lit_streams_off;
        const uint8_t *payload = input + d->src_off + d->lit_off + so;
        uint32_t plen = d->lit_comp_size - so;
        uint8_t *dst = lit_scratch + d->lit_buf_off;
        uint32_t mb = slot->max_bits, regen = d->regen_size;
        if (d->nstreams == 4) {
            uint32_t j1 = 0, j2 = 0, j3 = 0;
            if (plen < 6) { err = B200Z_ERR_LIT_MISSING_BYTES_FOR_JUMP_HEADER; }
            else {
                j1 = payload[0] | (payload[1] << 8); j2 = j1 + (payload[2] | (payload[3] << 8)); j3 = j2 + (payload[4] | (payload[5] << 8));
                if (plen - 6 < j3) err = B200Z_ERR_LIT_MISSING_BYTES_FOR_LITERALS;
            }
            if (!err) {
                const uint8_t *s0 = payload + 6;
                uint32_t S = (regen + 3) >> 2;
                uint32_t off[5] = {0, j1, j2, j3, plen - 6};
                // fast path: the standard split -- streams 0..2 regenerate S bytes, stream 3 the rest
                if (regen >= 3 * S) {
                    uint32_t cap = k < 3 ? S : regen - 3 * S;
                    uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(smem_huf + HUF_BLOCKS_PER_CTA * HUF_SMEM_PER_BLOCK + lane * RING_STRIDE);
                    irregular = !huf_stream_fast(tsym, tnb, mb, s0 + off[k], off[k + 1] - off[k], dst + k * S, cap, ring_addr);
                } else irregular = true;
                // any anomaly in the group -> lane 0 of the group replays the block with the reference's exact semantics
                uint32_t gmask = 0xFu << (lane & 28u);
                bool any = __any_sync(gmask, irregular);
                if (any && k == 0) {
                    uint32_t total = 0;
                    for (uint32_t s = 0; s < 4 && !err; s++) {
                        uint32_t c = 0;
                        uint32_t lim = total < regen ? regen - total : 0;
                        int r = huf_stream2(tsym, tnb, mb, s0 + off[s], off[s + 1] - off[s], dst + (total < regen ? total : regen), lim, 0xFFFFFFFFu, c);
                        if (r == 3) err = B200Z_ERR_LIT_EXTRA_PADDING;
                        else if (r == 1) err = B200Z_ERR_LIT_BITSTREAM_READ_MISMATCH;
                        total += c;
                    }
                    if (!err && total != regen) err = B200Z_ERR_LIT_DECODED_LITERAL_COUNT_MISMATCH;
                }
            }
        } else if (k == 0) {
            // single stream: no exact-landing check (literals_section_decoder.rs:143-147), only the total count
            rc = huf_stream2(tsym, tnb, mb, payload, plen, dst, regen, 0xFFFFFFFFu, count);
            if (rc == 3) err = B200Z_ERR_LIT_EXTRA_PADDING;
            else if (count != regen) err = B200Z_ERR_LIT_DECODED_LITERAL_COUNT_MISMATCH;
        }
    }
    if (active && k == 0 && err) aux[b].status = mk_status(err, B200Z_STAGE_LITERALS);
}

// ------------------------------------------------------------------------------------------------------------
// k_fse: sequences.  One lane per block, FSE_LANES blocks per one-warp CTA; the (LL + ML + OF) 16-bit LUTs of the
// CTA's blocks are staged into shared memory (2.5 KiB per block), code -> (baseline, extra bits) comes from two small
// shared LUTs, the reversed bitstream is read through PosRing (one 64-bit window per sequence), and sequences are
// written four at a time as three 16-byte vectors.  A warp alone on its scheduler is bound by the 16-lane integer
// pipe (2 cycles per warp instruction), not by dependencies: the step is written for instruction count.
// ------------------------------------------------------------------------------------------------------------
#ifndef B200Z_FSE_CHAINS
#define B200Z_FSE_CHAINS 1
#endif
constexpr uint32_t FSE_CHAINS = B200Z_FSE_CHAINS;            // blocks per lane, decoded interleaved
#ifndef B200Z_FSE_LANES
#define B200Z_FSE_LANES 16
#endif
constexpr uint32_t FSE_LANES = B200Z_FSE_LANES;              // lanes of the warp that carry blocks
constexpr uint32_t FSE_BLOCKS_PER_CTA = FSE_LANES * FSE_CHAINS;
constexpr uint32_t FSE_TAB_U16 = 512 + 512 + 256;   // LL, ML, OF entries per block
#ifndef B200Z_FSE_PUBLISH
#define B200Z_FSE_PUBLISH 128u   // sequences between two progress publications (power of two, multiple of 4)
#endif

__constant__ uint32_t c_ll_base[36] = {0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,18,20,22,24,28,32,40,48,64,128,256,512,1024,2048,4096,8192,16384,32768,65536};
__constant__ uint8_t c_ll_bits[36] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,6,7,8,9,10,11,12,13,14,15,16};
__constant__ uint32_t c_ml_base[53] = {3,4,5,6,7,8,9,10,11,12,13,14,15,16,17,18,19,20,21,22,23,24,25,26,27,28,29,30,31,32,33,34,35,37,39,41,43,47,51,59,67,83,99,131,259,515,1027,2051,4099,8195,16387,32771,65539};
__constant__ uint8_t c_ml_bits[53] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,4,5,7,8,9,10,11,12,13,14,15,16};

// do_offset_history (sequence_execution.rs:59-118): offset_value + literal length -> actual offset, history updated
__device__ __forceinline__ uint32_t offset_history_step(uint32_t of, uint32_t ll, uint32_t &h0, uint32_t &h1, uint32_t &h2) {
    uint32_t actual;
    if (ll > 0) {
        if (of == 1) actual = h0;
        else if (of == 2) { actual = h1; h1 = h0; h0 = actual; }
        else if (of == 3) { actual = h2; h2 = h1; h1 = h0; h0 = actual; }
        else { actual = of - 3; h2 = h1; h1 = h0; h0 = actual; }
    } else {
        if (of == 1) { actual = h1; h1 = h0; h0 = actual; }
        else if (of == 2) { actual = h2; h2 = h1; h1 = h0; h0 = actual; }
        else if (of == 3) { actual = h0 ? h0 - 1 : 0; h2 = h1; h1 = h0; h0 = actual; }   // saturating_sub, :74
        else { actual = of - 3; h2 = h1; h1 = h0; h0 = actual; }
    }
    return actual;
}

// hand-off to k_exec (which may run concurrently): results first, fence, then the flag
__device__ __forceinline__ void fse_publish_progress(BlockAux *aux, uint32_t b, uint32_t nseq_done) {
    __threadfence();
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(&aux[b].progress), "r"(nseq_done) : "memory");
}
__device__ __forceinline__ void fse_publish_ready(BlockAux *aux, uint32_t b) {
    __threadfence();
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(&aux[b].ready), "r"(1u) : "memory");
}

struct FseState {
    uint32_t e;   // current 16-bit entry
    __device__ __forceinline__ uint32_t sym() const { return e >> 10; }
    // num_bits and base_line out of the compact entry (b200z_types.h)
    __device__ __forceinline__ void decode(uint32_t log, uint32_t &nb, uint32_t &base) const {
        uint32_t f = e & 1023u;
        uint32_t h = 31u - (uint32_t)__clz((int)f);
        nb = log - h;
        base = (f ^ (1u << h)) << nb;
    }
};

// One block's sequence decode on the fast path: everything a chain carries between steps.  A lane runs FSE_CHAINS of
// them interleaved -- the chains are independent, so the second one's instructions fill the dependency stalls of the
// first (one warp per scheduler: there is nobody else to issue).
struct FseChain {
    // per block
    uint32_t b; const BlockDesc *d; bool active, run, bad; uint32_t st_seq;
    const FseTab *tl, *to, *tm;
    uint32_t logL, logM, logO, qTL, qTM, qTO;   // accuracy logs; shared-memory table addresses biased by -2^log entries
    uint32_t *out; uint32_t nseq;
    // running
    PosRing br;
    uint32_t eL, eM, eO, h0, h1, h2;   // h*: repeat-offset history, symbolic (b200z_types.h seq_sym_*)
    uint32_t out_end, lit_end, ovf;    // prefix sums of ll + ml and of ll; OR of all their values (bit 31 = reached 2^31)
    uint32_t flags, max_of, max_x, i;
};

__device__ __forceinline__ uint32_t fse_lds16(uint32_t addr) { uint16_t w; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(w) : "r"(addr) : "memory"); return w; }

// one sequence (sequence_section_decoder.rs:168-207); `update` = not the block's last sequence.  The record written is
// {out_end, lit_end, offset}: running sums of ll + ml and of ll (so that the execution kernels can place any sequence
// without a scan) and the offset after do_offset_history on symbolic history values.
__device__ __forceinline__ void fse_step(FseChain &c, uint32_t qLL, uint32_t qML, uint32_t &o_ll, uint32_t &o_ml, uint32_t &o_of, bool update) {
    uint32_t hi, lo;
    c.br.window(hi, lo);
    const uint32_t cL = c.eL >> 10, cM = c.eM >> 10, cO = c.eO >> 10;
    const uint32_t vL = lds32(qLL + (cL << 2)), vM = lds32(qML + (cM << 2));   // base | extra_bits << 24
    const uint32_t xL = vL >> 24, xM = vM >> 24, xO = cO;
    c.max_of = max(c.max_of, cO);   // offset codes >= 30 are checked per group (LL/ML codes are capped by table construction, scratch.rs:36-40)
    // extra bits: OF, ML, LL (get_bits_triple, sequence_section_decoder.rs:185)
    const uint32_t xsum = xO + xM + xL;
    c.max_x = max(c.max_x, xsum);   // > 38 extra bits in one sequence (the 64-bit window also has to hold the 26 state bits): not for
                                    // this path, checked per group.  (Far offsets with long lengths -- 1 MiB+ windows -- stay on this path.)
    const uint32_t t1 = fsl_c(lo, hi, xO), t2 = shl_c(t1, xM);   // the window below the offset bits: ML and LL extra bits (<= 32 together)
    const uint32_t obits = shr_c(hi, 32u - xO), ml_add = shr_c(t1, 32u - xM), ll_add = shr_c(t2, 32u - xL);
    uint32_t offset = obits + (1u << (cO & 31u));
    const uint32_t ll = (vL & 0xFFFFFFu) + ll_add, ml = (vM & 0xFFFFFFu) + ml_add;
    c.lit_end += ll; c.out_end += ll + ml;
    c.ovf |= c.out_end | c.lit_end;
    {   // do_offset_history (sequence_execution.rs:59-118), branch-free, on symbolic history values
        const bool rep = offset <= 3u;
        const uint32_t r = offset - 1u + (ll == 0u ? 1u : 0u);   // 0..3 when rep
        const uint32_t h0m1 = (c.h0 >> SEQ_SYM_SHIFT) ? c.h0 + 1u : c.h0 - (c.h0 != 0u ? 1u : 0u);   // saturating_sub (:74); symbols count the decrements
        uint32_t cand = c.h0;
        cand = r == 1u ? c.h1 : cand;
        cand = r == 2u ? c.h2 : cand;
        cand = r == 3u ? h0m1 : cand;
        const uint32_t actual = rep ? cand : offset - 3u;
        const bool keep2 = rep && r <= 1u, keep1 = rep && r == 0u;
        c.h2 = keep2 ? c.h2 : c.h1;
        c.h1 = keep1 ? c.h1 : c.h0;
        c.h0 = actual;
        offset = actual;
    }
    o_ll = c.out_end; o_ml = c.lit_end; o_of = offset;
    if (update) {   // state updates LL, ML, OF (:198-207); compact entries (b200z_types.h): nb = log - floor(log2 f)
        const uint32_t fL = c.eL & 1023u, fM = c.eM & 1023u, fO = c.eO & 1023u;
        const uint32_t nbL = c.logL - bfind32(fL), nbM = c.logM - bfind32(fM), nbO = c.logO - bfind32(fO);
        // the bits below the extra bits (up to 26 are used): a clamped funnel shift covers xsum <= 32, the rest comes out of lo
        uint32_t u0 = fsl_c(lo, hi, xsum);
        if (xsum > 32u) u0 = shl_c(lo, xsum - 32u);   // (rare; predicated, off the common dependency chain)
        const uint32_t u1 = shl_c(u0, nbL), u2 = shl_c(u1, nbM);
        const uint32_t aL = shr_c(u0, 32u - nbL), aM = shr_c(u1, 32u - nbM), aO = shr_c(u2, 32u - nbO);
        c.eL = fse_lds16(c.qTL + (((fL << nbL) + aL) << 1));
        c.eM = fse_lds16(c.qTM + (((fM << nbM) + aM) << 1));
        c.eO = fse_lds16(c.qTO + (((fO << nbO) + aO) << 1));
        c.br.P -= (int32_t)(xsum + nbL + nbM + nbO);
    } else c.br.P -= (int32_t)xsum;
}
__device__ __forceinline__ void fse_group_end(FseChain &c, const uint32_t (&stage)[12]) {
    c.flags |= (uint32_t)(c.br.P < 0) | (uint32_t)(c.max_x > 38u) | ((c.max_of + 2u) >> 5);   // bits_remaining only decreases: one check per group is equivalent
    uint4 *o4 = reinterpret_cast<uint4 *>(c.out + 3 * c.i);
    o4[0] = make_uint4(stage[0], stage[1], stage[2], stage[3]);
    o4[1] = make_uint4(stage[4], stage[5], stage[6], stage[7]);
    o4[2] = make_uint4(stage[8], stage[9], stage[10], stage[11]);
}

// the exact path (rare): the reference's control flow, one check at a time, for one block
__device__ __noinline__ void fse_exact_block(const BlockDesc *d, BlockAux *aux, uint32_t b, const uint8_t *input, uint32_t *seq_scratch,
                                             const uint16_t *TL, const uint16_t *TM, const uint16_t *TO, const FseTab *tl, const FseTab *to, const FseTab *tm,
                                             const uint32_t *s_ll_base, const uint32_t *s_ml_base, const uint8_t *s_ll_bits, const uint8_t *s_ml_bits, uint32_t st_seq) {
    // Emits the same prefix-form records as the fast path but with RAW offset_values (full 32-bit range: an offset code
    // >= 30 cannot be told from a symbol) and flags the block AUX_RAW_OFFSETS: the warp-per-frame execution kernel then
    // runs do_offset_history itself, sequence by sequence.
    uint32_t err = 0;
    uint32_t out_end = 0, lit_end = 0, ovf = 0;
    {
        const uint8_t *src = input + d->src_off + aux[b].seq_bits_off;
        uint32_t len = d->src_size - aux[b].seq_bits_off;
        HufBits br;
        FseState sl{0}, so{0}, sm{0};
        uint32_t logL = 0, logM = 0, logO = 0;
        if (!br.init(src, len)) err = B200Z_ERR_SEQ_EXTRA_PADDING;
        // init order LL, OF, ML (sequence_section_decoder.rs:164-166); an RLE'd component reads 0 bits
        if (!err) { if (!tl || !tl->valid) err = B200Z_ERR_FSE_TABLE_IS_UNINITIALIZED; else { logL = tl->log; br.refill(); uint32_t i = logL ? br.hi >> (32u - logL) : 0u; br.skip(logL); sl.e = TL[i]; } }
        if (!err) { if (!to || !to->valid) err = B200Z_ERR_FSE_TABLE_IS_UNINITIALIZED; else { logO = to->log; br.refill(); uint32_t i = logO ? br.hi >> (32u - logO) : 0u; br.skip(logO); so.e = TO[i]; } }
        if (!err) { if (!tm || !tm->valid) err = B200Z_ERR_FSE_TABLE_IS_UNINITIALIZED; else { logM = tm->log; br.refill(); uint32_t i = logM ? br.hi >> (32u - logM) : 0u; br.skip(logM); sm.e = TM[i]; } }
        uint32_t *out = seq_scratch + d->seq_buf_off * 3;   // 16-byte aligned: the planner rounds seq_buf_off to 4 sequences
        const uint32_t nseq = d->nseq;
        uint32_t stage[12];
        // one sequence; `last` suppresses the state update exactly like `target.len() < num_sequences` (:198)
        auto one = [&](uint32_t &ll, uint32_t &ml, uint32_t &offset, bool last) {
            const uint32_t ll_code = sl.sym(), ml_code = sm.sym(), of_code = so.sym();
            if (ll_code > 35 || ml_code > 52) { err = B200Z_ERR_REFERENCE_WOULD_PANIC; return; }  // unreachable!: tables cap the symbols
            if (of_code > 31) { err = B200Z_ERR_SEQ_UNSUPPORTED_OFFSET; return; }
            const uint32_t ll_bits = s_ll_bits[ll_code], ml_bits = s_ml_bits[ml_code];
            uint32_t nbL, nbM, nbO, baseL, baseM, baseO;
            sl.decode(logL, nbL, baseL); sm.decode(logM, nbM, baseM); so.decode(logO, nbO, baseO);
            // extra bits in the order OF, ML, LL (get_bits_triple, :185); then the state updates LL, ML, OF (:198-207)
            br.refill();
            uint32_t obits = of_code ? br.hi >> (32u - of_code) : 0u;
            br.skip(of_code);
            br.refill();
            uint32_t ml_add = ml_bits ? br.hi >> (32u - ml_bits) : 0u; br.skip(ml_bits);
            uint32_t ll_add = ll_bits ? br.hi >> (32u - ll_bits) : 0u; br.skip(ll_bits);
            offset = obits + (1u << of_code);
            const uint32_t llv = s_ll_base[ll_code] + ll_add, mlv = s_ml_base[ml_code] + ml_add;
            lit_end += llv; out_end += llv + mlv; ovf |= out_end | lit_end;
            ll = out_end; ml = lit_end;   // the record is {out_end, lit_end, raw offset}
            if (!last) {
                br.refill();
                uint32_t aL = nbL ? br.hi >> (32u - nbL) : 0u; br.skip(nbL);
                uint32_t aM = nbM ? br.hi >> (32u - nbM) : 0u; br.skip(nbM);
                uint32_t aO = nbO ? br.hi >> (32u - nbO) : 0u; br.skip(nbO);
                sl.e = TL[baseL + aL]; sm.e = TM[baseM + aM]; so.e = TO[baseO + aO];
            }
            if (br.p < 0) err = B200Z_ERR_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES;
        };
        uint32_t i = 0;
        for (; i + 4 < nseq && !err; i += 4) {   // groups of four, none of them the last sequence
#pragma unroll
            for (int q = 0; q < 4; q++) { if (!err) one(stage[3 * q], stage[3 * q + 1], stage[3 * q + 2], false); }
            if (!err) {
                uint4 *o4 = reinterpret_cast<uint4 *>(out + 3 * i);
                o4[0] = make_uint4(stage[0], stage[1], stage[2], stage[3]);
                o4[1] = make_uint4(stage[4], stage[5], stage[6], stage[7]);
                o4[2] = make_uint4(stage[8], stage[9], stage[10], stage[11]);
            }
        }
        for (; i < nseq && !err; i++) {
            uint32_t ll = 0, ml = 0, of = 0;
            one(ll, ml, of, i + 1 == nseq);
            if (!err || err == B200Z_ERR_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES) { out[3 * i] = ll; out[3 * i + 1] = ml; out[3 * i + 2] = of; }
        }
        if (!err && br.p > 0) err = B200Z_ERR_SEQ_EXTRA_BITS;
        if (err) st_seq = mk_status(err, B200Z_STAGE_SEQUENCES);
    }
    aux[b].pad = st_seq;
    aux[b].sum_ll = lit_end;
    aux[b].flags = AUX_RAW_OFFSETS | ((ovf >> 31) ? AUX_WIDE : 0u);
    aux[b].out_size = (ovf >> 31) ? 0xffffffffu : out_end - lit_end + d->regen_size;   // sum of ml + regenerated literals
}

#ifdef B200Z_PROBE
// Development probe (profiles/variants.sh probe "-DB200Z_PROBE", profiles/probe_overlap.py): device timestamps of the k_fse / k_exec pair.
// [0] first k_fse CTA start, [1] last k_fse CTA end, [2] first k_exec warp start, [3] last k_exec warp end, [4] last k_exec warp start,
// [5] first k_exec warp end (globaltimer, ns).  Not part of the shipped library.
__device__ unsigned long long g_probe[8];
__device__ __forceinline__ unsigned long long probe_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
extern "C" int b200z_probe_read(unsigned long long *out, int reset) {
    if (out && cudaMemcpyFromSymbol(out, g_probe, sizeof(unsigned long long) * 8) != cudaSuccess) return 1;
    if (reset) {
        const unsigned long long init[8] = {~0ull, 0, ~0ull, 0, 0, ~0ull, 0, 0};
        if (cudaMemcpyToSymbol(g_probe, init, sizeof init) != cudaSuccess) return 1;
    }
    return 0;
}
#endif
__global__ void __launch_bounds__(32) k_fse(const BlockDesc *__restrict__ descs, BlockAux *__restrict__ aux, const uint8_t *__restrict__ input,
                                          uint32_t *__restrict__ seq_scratch, uint32_t nblocks, const uint32_t *__restrict__ order) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // this CTA is resident: k_exec may follow (launch_pipeline_overlapped)
#ifdef B200Z_PROBE
    if (threadIdx.x == 0) atomicMin(&g_probe[0], probe_now());
#endif
    extern __shared__ __align__(16) uint8_t smem_fse[];
    uint16_t *tabs = reinterpret_cast<uint16_t *>(smem_fse);
    uint32_t *s_ll_base = reinterpret_cast<uint32_t *>(smem_fse + FSE_BLOCKS_PER_CTA * FSE_TAB_U16 * 2);
    uint32_t *s_ml_base = s_ll_base + 36;
    uint8_t *s_ll_bits = reinterpret_cast<uint8_t *>(s_ml_base + 53);
    uint8_t *s_ml_bits = s_ll_bits + 36;
    uint32_t *s_ll = reinterpret_cast<uint32_t *>(smem_fse + FSE_BLOCKS_PER_CTA * FSE_TAB_U16 * 2 + 512);   // base | bits << 24
    uint32_t *s_ml = s_ll + 36;
    uint8_t *s_ring = smem_fse + FSE_BLOCKS_PER_CTA * FSE_TAB_U16 * 2 + 1024;                                // FSE_BLOCKS_PER_CTA x RING_STRIDE
    const uint32_t lane = threadIdx.x;
    for (uint32_t i = lane; i < 36; i += 32) { s_ll_base[i] = c_ll_base[i]; s_ll_bits[i] = c_ll_bits[i]; s_ll[i] = c_ll_base[i] | ((uint32_t)c_ll_bits[i] << 24); }
    for (uint32_t i = lane; i < 53; i += 32) { s_ml_base[i] = c_ml_base[i]; s_ml_bits[i] = c_ml_bits[i]; s_ml[i] = c_ml_base[i] | ((uint32_t)c_ml_bits[i] << 24); }

    FseChain ch[FSE_CHAINS];
#pragma unroll
    for (int k = 0; k < (int)FSE_CHAINS; k++) {
        FseChain &c = ch[k];
        c.b = blockIdx.x * FSE_BLOCKS_PER_CTA + FSE_CHAINS * lane + k;   // neighbouring blocks share a lane: similar lengths
        c.active = lane < FSE_LANES && c.b < nblocks;
        if (c.active && order) c.b = order[c.b];   // PipelineArgs::fse_order
        c.d = c.active ? &descs[c.b] : nullptr;
        c.st_seq = 0; c.run = false; c.bad = false;
        if (c.active) {
            c.st_seq = aux[c.b].pad;
            if (c.d->btype != BT_COMPRESSED) aux[c.b].out_size = c.d->raw_size;
            else if (!c.d->host_status && c.d->nseq == 0) aux[c.b].out_size = c.d->regen_size;
            c.run = c.d->btype == BT_COMPRESSED && !c.d->host_status && c.d->nseq != 0 && c.st_seq == 0;
        }
        c.tl = c.run ? c.d->ll : nullptr; c.to = c.run ? c.d->of : nullptr; c.tm = c.run ? c.d->ml : nullptr;
    }
    // ---- stage the tables of the CTA's blocks (warp-cooperative, 16-byte vectors); slot = FSE_CHAINS * lane + chain
    for (uint32_t j = 0; j < FSE_LANES; j++) {
#pragma unroll
        for (int k = 0; k < (int)FSE_CHAINS; k++) {
            const FseTab *pj[3];
            pj[0] = (const FseTab *)(uintptr_t)__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)ch[k].tl, j);
            pj[1] = (const FseTab *)(uintptr_t)__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)ch[k].tm, j);
            pj[2] = (const FseTab *)(uintptr_t)__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)ch[k].to, j);
            uint16_t *dstj = tabs + (FSE_CHAINS * j + k) * FSE_TAB_U16;
            const uint32_t offs[3] = {0, 512, 1024};
#pragma unroll
            for (int t = 0; t < 3; t++) {
                if (!pj[t] || !pj[t]->valid) continue;
                uint32_t n16 = ((2u << pj[t]->log) + 15) >> 4;   // bytes / 16
                if (t == 2 && n16 > 32) n16 = 32;
                if (n16 > 64) n16 = 64;
                const uint4 *s4 = reinterpret_cast<const uint4 *>(pj[t]->e);
                uint4 *d4 = reinterpret_cast<uint4 *>(dstj + offs[t]);
                for (uint32_t i = lane; i < n16; i += 32) d4[i] = s4[i];
            }
        }
    }
    __syncwarp();
    uint32_t qLL = (uint32_t)__cvta_generic_to_shared(s_ll), qML = (uint32_t)__cvta_generic_to_shared(s_ml);
    asm volatile("" : "+r"(qLL), "+r"(qML));

    // ---------------- fast path: branch-free steps; anything unusual (bad code, > 32 extra bits in one sequence,
    // under/over-run, uninitialised table) sets `bad` and the block is decoded again by the exact path below.
#pragma unroll
    for (int k = 0; k < (int)FSE_CHAINS; k++) {
        FseChain &c = ch[k];
        if (!c.run) { c.bad = false; continue; }
        const uint32_t slot = FSE_CHAINS * lane + k;
        const uint8_t *src = input + c.d->src_off + aux[c.b].seq_bits_off;
        const uint32_t len = c.d->src_size - aux[c.b].seq_bits_off;
        const uint16_t *TL = tabs + slot * FSE_TAB_U16;
        const uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(s_ring + slot * RING_STRIDE) + 16u;   // slot 0; the mirror slot sits below
        c.bad = !c.br.init(src, len, ring_addr) || !c.tl || !c.tl->valid || !c.to || !c.to->valid || !c.tm || !c.tm->valid;
        if (!c.bad) c.bad = c.tl->log > 9u || c.tm->log > 9u || c.to->log > 8u;   // never true for a built table: the staged copies are sized for these
        c.flags = 0; c.max_of = 0; c.max_x = 0; c.i = 0; c.out_end = 0; c.lit_end = 0; c.ovf = 0;
        c.nseq = c.d->nseq;
        c.h0 = 1u << SEQ_SYM_SHIFT; c.h1 = 2u << SEQ_SYM_SHIFT; c.h2 = 3u << SEQ_SYM_SHIFT;   // "slot k at the block's start"
        c.out = seq_scratch + c.d->seq_buf_off * 3;
        if (!c.bad) {
            c.logL = c.tl->log; c.logM = c.tm->log; c.logO = c.to->log;
            const uint32_t aTL = (uint32_t)__cvta_generic_to_shared(TL), aTM = aTL + 1024u, aTO = aTL + 2048u;
            c.qTL = aTL - (2u << c.logL); c.qTM = aTM - (2u << c.logM); c.qTO = aTO - (2u << c.logO);
            // initial states LL, OF, ML (sequence_section_decoder.rs:164-166)
            uint32_t hi, lo;
            c.br.window(hi, lo);
            const uint32_t t1 = shl_c(hi, c.logL), t2 = shl_c(t1, c.logO);
            c.eL = fse_lds16(aTL + (shr_c(hi, 32u - c.logL) << 1));
            c.eO = fse_lds16(aTO + (shr_c(t1, 32u - c.logO) << 1));
            c.eM = fse_lds16(aTM + (shr_c(t2, 32u - c.logM) << 1));
            c.br.P -= (int32_t)(c.logL + c.logO + c.logM);
        }
    }
    // joint loop: groups of four sequences of every chain, step by step in turn
    {
        bool joint = true;
        uint32_t nmin = 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < (int)FSE_CHAINS; k++) { joint = joint && ch[k].run && !ch[k].bad; nmin = min(nmin, ch[k].run ? ch[k].nseq : 0u); }
        if (FSE_CHAINS > 1 && joint) {
            uint32_t stage[FSE_CHAINS][12];
            uint32_t i = 0, anyflag = 0;
            for (; i + 4 < nmin; i += 4) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
#pragma unroll
                    for (int k = 0; k < (int)FSE_CHAINS; k++) fse_step(ch[k], qLL, qML, stage[k][3 * q], stage[k][3 * q + 1], stage[k][3 * q + 2], true);
                    if (q & 1) {
#pragma unroll
                        for (int k = 0; k < (int)FSE_CHAINS; k++) ch[k].br.service();
                    }
                }
#pragma unroll
                for (int k = 0; k < (int)FSE_CHAINS; k++) { ch[k].i = i; fse_group_end(ch[k], stage[k]); anyflag |= ch[k].flags; }
                if (anyflag) { i += 4; break; }
            }
#pragma unroll
            for (int k = 0; k < (int)FSE_CHAINS; k++) ch[k].i = i;
        }
    }
    // each chain on its own: the rest of its groups, then its last sequences one at a time
#pragma unroll
    for (int k = 0; k < (int)FSE_CHAINS; k++) {
        FseChain &c = ch[k];
        if (!c.run || c.bad) continue;
        if (!c.flags) {
            uint32_t stage[12];
            for (; c.i + 4 < c.nseq; c.i += 4) {
#pragma unroll
                for (int q = 0; q < 4; q++) { fse_step(c, qLL, qML, stage[3 * q], stage[3 * q + 1], stage[3 * q + 2], true); if (q & 1) c.br.service(); }
                fse_group_end(c, stage);
                if (c.flags) break;
                if (((c.i + 4) & (B200Z_FSE_PUBLISH - 1u)) == 0) fse_publish_progress(aux, c.b, c.i + 4);   // the fence costs ~1 us
            }
        }
        if (!c.flags) {
            for (; c.i < c.nseq; c.i++) {
                uint32_t ll, ml, of;
                fse_step(c, qLL, qML, ll, ml, of, c.i + 1 < c.nseq);
                c.br.service();
                c.flags |= (uint32_t)(c.br.P < 0) | (uint32_t)(c.max_x > 38u) | ((c.max_of + 2u) >> 5);
                c.out[3 * c.i] = ll; c.out[3 * c.i + 1] = ml; c.out[3 * c.i + 2] = of;
            }
        }
        c.bad = c.flags != 0 || c.br.P != 0;
        if (!c.bad) {
            aux[c.b].pad = 0;
            aux[c.b].hist_after[0] = c.h0; aux[c.b].hist_after[1] = c.h1; aux[c.b].hist_after[2] = c.h2;
            aux[c.b].sum_ll = c.lit_end;
            aux[c.b].flags = (c.ovf >> 31) ? AUX_WIDE : 0u;
            aux[c.b].out_size = (c.ovf >> 31) ? 0xffffffffu : c.out_end - c.lit_end + c.d->regen_size;   // sum of ml + regenerated literals
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    // verdicts; blocks the fast path gave up on are decoded again by the exact path
#pragma unroll
    for (int k = 0; k < (int)FSE_CHAINS; k++) {
        FseChain &c = ch[k];
        if (!c.active) continue;
        if (!c.run) { aux[c.b].pad = c.st_seq; continue; }
        if (!c.bad) continue;
        const uint16_t *TL = tabs + (FSE_CHAINS * lane + k) * FSE_TAB_U16;
        fse_exact_block(c.d, aux, c.b, input, seq_scratch, TL, TL + 512, TL + 1024, c.tl, c.to, c.tm, s_ll_base, s_ml_base, s_ll_bits, s_ml_bits, c.st_seq);
    }
    // hand-off: the block's records, verdict and sizes are in memory
#pragma unroll
    for (int k = 0; k < (int)FSE_CHAINS; k++)
        if (ch[k].active) fse_publish_ready(aux, ch[k].b);
#ifdef B200Z_PROBE
    if (threadIdx.x == 0) atomicMax(&g_probe[1], probe_now());
#endif
}

// ------------------------------------------------------------------------------------------------------------
// k_exec: LZ77 execution.  One warp per frame, blocks in order, 64 sequences per step.
//
// Fast path (per batch of 64 sequences, lane j = sequences 2j and 2j + 1): one warp scan gives every sequence its
// literal and match positions; a bitmask of sequence ends in shared memory lets each OUTPUT byte find its owner
// with one popc, an 8-byte record per sequence tells it where it comes from; the batch's bytes are then produced
// row by row (32 consecutive bytes = one coalesced store), four rows' loads in flight: literal bytes and match
// bytes whose source is final first, then the few match bytes whose source lies inside the same four rows,
// looping inside a row until it is complete (sources always precede destinations, so the lowest pending byte is
// always ready).  Overlapping matches use source = start + (k mod offset), the byte-order-preserving form of
// repeat_in_chunks (decode_buffer.rs:113-141).  Anything unusual in a batch (dictionary reach, zero offsets,
// literal under-run, capacity, more than EXEC_TMAX bytes) sends that batch to the exact sequential path below,
// which is execute_sequences / DecodeBuffer::repeat statement by statement.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_copy(uint8_t *dst, const uint8_t *src, uint32_t n, uint32_t lane) {
    for (uint32_t k = lane; k < n; k += 32) dst[k] = src[k];
}
__device__ __forceinline__ void warp_fill(uint8_t *dst, uint8_t v, uint32_t n, uint32_t lane) {
    for (uint32_t k = lane; k < n; k += 32) dst[k] = v;
}
__device__ __forceinline__ void warp_match(uint8_t *dst, const uint8_t *src, uint32_t n, uint32_t off, uint32_t lane) {
    if (off >= n) { for (uint32_t k = lane; k < n; k += 32) dst[k] = src[k]; }
    else { for (uint32_t k = lane; k < n; k += 32) dst[k] = src[k % off]; }
}

struct ExecState {
    uint32_t h0, h1, h2;
    uint64_t produced, counter, drained, cap;
    uint32_t litpos;
};
struct LitSrc { const uint8_t *p; uint32_t rle; uint8_t byte; uint32_t regen; };

// exact sequential execution of up to 32 sequences held one per lane (my_ll/my_ml/my_of); `resolved` = offsets
// already went through do_offset_history.  Returns 0 or an error code.
#ifndef B200Z_EXEC_PER_LANE
#define B200Z_EXEC_PER_LANE 2
#endif
constexpr uint32_t EXEC_PER_LANE = B200Z_EXEC_PER_LANE;      // consecutive sequences a lane holds (even)
constexpr uint32_t EXEC_BATCH = 32 * EXEC_PER_LANE;         // sequences per batch
// Sequence j of the batch lives in lane j / EXEC_PER_LANE, slot j % EXEC_PER_LANE.
__device__ __forceinline__ uint32_t exec_pick(const uint32_t (&v)[EXEC_PER_LANE], uint32_t slot) {
    uint32_t r = v[0];
#pragma unroll
    for (uint32_t k = 1; k < EXEC_PER_LANE; k++) r = slot == k ? v[k] : r;
    return r;
}
__device__ uint32_t exec_batch_exact(ExecState &st, const LitSrc &lit, const FrameDesc &fd, uint8_t *out, uint32_t nb, const uint32_t (&lls)[EXEC_PER_LANE],
                                     const uint32_t (&mls)[EXEC_PER_LANE], const uint32_t (&ofs)[EXEC_PER_LANE], bool resolved, uint32_t lane) {
    for (uint32_t j = 0; j < nb; j++) {
        const uint32_t slot = j % EXEC_PER_LANE, src_lane = j / EXEC_PER_LANE;
        uint32_t ll = __shfl_sync(0xffffffffu, exec_pick(lls, slot), src_lane), ml = __shfl_sync(0xffffffffu, exec_pick(mls, slot), src_lane),
                 of = __shfl_sync(0xffffffffu, exec_pick(ofs, slot), src_lane);
        if (ll > 0) {
            if ((uint64_t)st.litpos + ll > lit.regen) return B200Z_ERR_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE;
            if (st.produced + ll > st.cap) return B200Z_ERR_TARGET_TOO_SMALL;
            if (lit.rle) warp_fill(out + st.produced, lit.byte, ll, lane); else warp_copy(out + st.produced, lit.p + st.litpos, ll, lane);
            st.litpos += ll; st.produced += ll; st.counter += ll;
        }
        uint32_t actual = resolved ? of : offset_history_step(of, ll, st.h0, st.h1, st.h2);
        if (actual == 0) return B200Z_ERR_EXEC_ZERO_OFFSET;
        if (ml > 0) {
            if (st.produced + ml > st.cap) return B200Z_ERR_TARGET_TOO_SMALL;
            __syncwarp();
            uint64_t buf_len = st.produced - st.drained;
            if ((uint64_t)actual > buf_len) {
                // repeat_from_dict (decode_buffer.rs:143-179)
                if (st.counter <= fd.window_size) {
                    uint64_t from_dict = (uint64_t)actual - buf_len;
                    if (from_dict > fd.dict_len) return B200Z_ERR_EXEC_NOT_ENOUGH_BYTES_IN_DICTIONARY;
                    if (from_dict < ml) {
                        warp_copy(out + st.produced, fd.dict + fd.dict_len - from_dict, (uint32_t)from_dict, lane);
                        st.produced += from_dict; st.counter += from_dict;
                        __syncwarp();
                        uint32_t rest = ml - (uint32_t)from_dict;
                        uint64_t bl2 = st.produced - st.drained;  // repeat(self.buffer.len(), rest): from the buffer start
                        warp_match(out + st.produced, out + st.drained, rest, bl2 > 0xffffffffull ? 0xffffffffu : (uint32_t)bl2, lane);
                        st.produced += rest; st.counter += rest;
                    } else {
                        warp_copy(out + st.produced, fd.dict + fd.dict_len - from_dict, ml, lane);
                        st.produced += ml;  // sic: total_output_counter not advanced on this branch (:166-171)
                    }
                } else return B200Z_ERR_EXEC_OFFSET_TOO_BIG;
            } else {
                warp_match(out + st.produced, out + st.produced - actual, ml, actual, lane);
                st.produced += ml; st.counter += ml;
            }
            __syncwarp();
        }
    }
    return 0;
}

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint2 ld_cg_u32x2(const uint32_t *p) {
    uint2 v;
    asm volatile("ld.global.cg.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Block-granular hand-off from k_fse (fse_publish_ready): k_exec may be launched as k_fse's programmatic dependent and then
// runs beside it; a frame's block is executed as soon as its sequence stage is over.  Bounded by wall clock (globaltimer),
// generously: the producer always shows up (all of k_fse's CTAs are resident before k_exec's first one, programmatic
// dependent launch), a timeout means the device is shared or being debugged -- it is reported as B200Z_ERR_CUDA for the
// frame instead of hanging the GPU.  Warp-uniform result.
__device__ __forceinline__ bool exec_wait_ready(const BlockAux *aux, uint32_t b, uint32_t lane) {
    uint32_t ok = 1;
    if (lane == 0) {
        if (ld_acquire_u32(&aux[b].ready) == 0u) {
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            for (;;) {
                __nanosleep(500);
                if (ld_acquire_u32(&aux[b].ready) != 0u) break;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 20000000000ull) { ok = 0; break; }   // 20 s
            }
        }
    }
    return __shfl_sync(0xffffffffu, ok, 0) != 0;
}

#ifndef B200Z_EXEC_WARPS
#define B200Z_EXEC_WARPS 4
#endif
constexpr uint32_t EXEC_WARPS = B200Z_EXEC_WARPS;
#ifndef B200Z_EXEC_TMAX
#define B200Z_EXEC_TMAX 8128
#endif
constexpr uint32_t EXEC_TMAX = B200Z_EXEC_TMAX;             // most bytes one batch may produce on the fast path (sizes the end-bit mask)
#ifndef B200Z_EXEC_CHUNK_ROWS
#define B200Z_EXEC_CHUNK_ROWS 4
#endif
#ifndef B200Z_EXEC_PREFETCH
#define B200Z_EXEC_PREFETCH 1
#endif
constexpr uint32_t EXEC_CHUNK_ROWS = B200Z_EXEC_CHUNK_ROWS;                    // rows (of 32 bytes) whose loads are in flight together
constexpr uint32_t EXEC_MASK_WORDS = (EXEC_TMAX + 31) / 32 + EXEC_CHUNK_ROWS;
#ifndef B200Z_EXEC_MINB
#define B200Z_EXEC_MINB 8
#endif

__global__ void __launch_bounds__(EXEC_WARPS * 32, B200Z_EXEC_MINB) k_exec(const BlockDesc *__restrict__ descs, const BlockAux *__restrict__ aux,
                                                        const FrameDesc *__restrict__ frames, FrameState *__restrict__ states,
                                                        const uint8_t *__restrict__ input, const uint8_t *__restrict__ lit_scratch,
                                                        const uint32_t *__restrict__ seq_scratch, uint8_t *__restrict__ output, uint64_t output_cap,
                                                        uint32_t nframes, uint32_t *__restrict__ resume, uint32_t frame_base) {
    __shared__ uint32_t s_mask[EXEC_WARPS][EXEC_MASK_WORDS];
    __shared__ __align__(16) uint2 s_recs[EXEC_WARPS][EXEC_BATCH];
    __shared__ ExecState s_saved[EXEC_WARPS];   // the state at the current block's start (kept out of the registers: read only on a rollback)
    const uint32_t f = frame_base + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const uint32_t lane = threadIdx.x & 31, lt = lanemask_lt();
    if (f >= nframes) return;
#ifdef B200Z_PROBE
    if (lane == 0) { const unsigned long long t = probe_now(); atomicMin(&g_probe[2], t); atomicMax(&g_probe[4], t); }
#endif
    uint32_t a_mask = (uint32_t)__cvta_generic_to_shared(s_mask[threadIdx.x >> 5]);   // this warp's bitmask of sequence ends
    uint32_t a_recs = (uint32_t)__cvta_generic_to_shared(s_recs[threadIdx.x >> 5]);   // this warp's per-sequence records
    asm volatile("" : "+r"(a_mask), "+r"(a_recs));   // keep both addresses in registers (ptxas would recompute them from %tid per chunk)
    const FrameDesc &fd = frames[f];
    // frames (or leading blocks of frames) that k_exec_cta already executed: resume[f] = first block left for this kernel
    const uint32_t first_bi = resume ? resume[f] : 0u;
    if (first_bi > fd.nblocks) return;   // nothing (left) for this launch: RESUME_SKIP, or k_exec_cta finished the frame
    FrameState fs = states[f];
    ExecState st;
    st.h0 = fs.hist[0]; st.h1 = fs.hist[1]; st.h2 = fs.hist[2];
    st.produced = fs.produced; st.counter = fs.counter; st.drained = fs.drained;
    st.cap = fd.out_cap;
    if (fd.out_off > output_cap) st.cap = 0; else if (st.cap > output_cap - fd.out_off) st.cap = output_cap - fd.out_off;
    uint8_t *out = output + fd.out_off;
    uint32_t status = fs.status, err_block = fs.error_block, blocks_done = fs.blocks_done;

    for (uint32_t bi = first_bi; bi < fd.nblocks && !status; bi++) {
        const uint32_t b = fd.first_block + bi;
        const BlockDesc &d = descs[b];
        // first error in the reference's order: header-level planner errors, literals, sequence header (planner),
        // sequence tables + decode, then execution
        uint32_t hs = d.host_status, hpos = hs >> 24;
        hs &= 0x00ffffffu;
        // k_fse may still be running (this kernel is its programmatic dependent).  The literals stage is complete (stream order);
        // the sequence stage of this block is over once BlockAux::ready is set -- until then its records are consumed as the
        // fast path of k_fse publishes them (BlockAux::progress).  Results of k_fse are read past the L1.
        const bool seq_block = d.btype == BT_COMPRESSED && d.nseq != 0 && !hs;
        bool known = !seq_block || __shfl_sync(0xffffffffu, lane == 0 ? ld_acquire_u32(&aux[b].ready) : 0u, 0) != 0u;   // the sequence stage's verdict is in
        const uint32_t ax_status = ld_cg_u32(&aux[b].status);
        uint32_t ax_pad = seq_block && known ? ld_cg_u32(&aux[b].pad) : 0u, ax_flags = seq_block && known ? ld_cg_u32(&aux[b].flags) : 0u;
        uint32_t bs = 0;
        if (hs && hpos == 1) bs = hs;
        else if (ax_status) bs = ax_status;
        else if (hs) bs = hs;
        else if (ax_pad) bs = ax_pad;
        // a block whose sequence stage failed executes nothing: in the reference decode_sequences completes before
        // execute_sequences starts (block_decoder.rs:176-183)
        if (bs) { status = bs; err_block = d.block_in_frame; break; }

        if (d.btype == BT_RAW) {
            if (st.produced + d.raw_size > st.cap) { status = mk_status(B200Z_ERR_TARGET_TOO_SMALL, B200Z_STAGE_DRAIN); err_block = d.block_in_frame; break; }
            warp_copy(out + st.produced, input + d.src_off, d.raw_size, lane);
            st.produced += d.raw_size;   // extend_from_reader: total_output_counter untouched (decode_buffer.rs:66-72)
        } else if (d.btype == BT_RLE) {
            if (st.produced + d.raw_size > st.cap) { status = mk_status(B200Z_ERR_TARGET_TOO_SMALL, B200Z_STAGE_DRAIN); err_block = d.block_in_frame; break; }
            warp_fill(out + st.produced, input[d.src_off], d.raw_size, lane);
            st.produced += d.raw_size;
        } else {
            LitSrc lit;
            lit.rle = 0; lit.byte = 0; lit.regen = d.regen_size;
            if (d.lit_type == LT_RAW) lit.p = input + d.src_off + d.lit_off;
            else if (d.lit_type == LT_RLE) { lit.p = nullptr; lit.rle = 1; lit.byte = input[d.src_off + d.lit_off]; }
            else lit.p = lit_scratch + d.lit_buf_off;
            // the block's start: where a sequence-stage error / a replay by the exact path rolls back to
            if (lane == 0) s_saved[threadIdx.x >> 5] = st;
            __syncwarp();
            uint32_t redo = 0;            // 1: sequence-stage error after records were consumed, 2: the records were rewritten with raw offsets
          exec_block_again:
            st = s_saved[threadIdx.x >> 5];
            st.litpos = 0;
            uint32_t e = 0;
            uint32_t avail = known ? 0xFFFFFFFFu : 0u;   // records that may be read
            // block-level descriptor fields used inside the batch loop are consumed here once: a first use inside the loop
            // would wait on a scoreboard shared with the record prefetch issued just before it (a full memory latency per batch)
            uint32_t resolved_u = (ax_flags & AUX_RAW_OFFSETS) ? 0u : 1u, nseq_u = d.nseq;
            const uint32_t *seqs = seq_scratch + d.seq_buf_off * 3;
            asm volatile("" : "+r"(resolved_u), "+r"(nseq_u), "+l"(seqs));
            const bool resolved = resolved_u != 0;
            __syncwarp();
            // A batch is EXEC_BATCH sequences, EXEC_PER_LANE consecutive ones per lane (contiguous 12-byte records in prefix
            // form {out_end, lit_end, of}: ll and ml are differences of neighbouring records); the next batch's records are
            // requested into L2 one batch ahead.
            constexpr uint32_t K = EXEC_PER_LANE;
            uint32_t carry_out = 0, carry_lit = 0;   // prefix sums at the end of the previous batch
            const uint32_t bh0 = st.h0, bh1 = st.h1, bh2 = st.h2;   // history at the block's start: what the symbols refer to
            for (uint32_t base = 0; base < nseq_u && !e; base += EXEC_BATCH) {
                const uint32_t nb = nseq_u - base < EXEC_BATCH ? nseq_u - base : EXEC_BATCH;
                if (avail < base + nb) {   // wait for k_fse: either these records, or the end of the block's sequence stage
                    uint32_t got = 0, fin = 0;
                    if (lane == 0) {
                        unsigned long long t0 = 0, t1;
                        for (uint32_t spins = 0;; spins++) {
                            fin = ld_acquire_u32(&aux[b].ready);
                            if (fin) break;
                            got = ld_acquire_u32(&aux[b].progress);
                            if (got >= base + nb) break;
                            __nanosleep(200);
                            if ((spins & 1023u) == 0) {
                                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                                if (t0 == 0) t0 = t1; else if (t1 - t0 > 20000000000ull) { fin = 2; break; }   // 20 s: see exec_wait_ready
                            }
                        }
                    }
                    fin = __shfl_sync(0xffffffffu, fin, 0); got = __shfl_sync(0xffffffffu, got, 0);
                    if (fin == 2) { e = B200Z_ERR_CUDA; break; }
                    if (fin) {
                        known = true; avail = 0xFFFFFFFFu;
                        ax_pad = ld_cg_u32(&aux[b].pad); ax_flags = ld_cg_u32(&aux[b].flags);
                        if (ax_pad) { redo = 1; break; }
                        if (ax_flags & AUX_RAW_OFFSETS) { redo = 2; break; }   // (the records consumed so far were symbolic: run the block again)
                    } else avail = got;
                }
                uint32_t lls[K], mls[K], ofs[K], pe_out[K], pe_lit[K];
                bool on[K];
                const uint32_t old_out = carry_out, old_lit = carry_lit;
                {
                    const uint32_t *sp = seqs + (uint64_t)(base + K * lane) * 3;
                    uint32_t raw[3 * K];
                    if (K * lane + K <= nb) {   // all my records exist: K * 12 contiguous bytes, 8-byte aligned
#pragma unroll
                        for (uint32_t k = 0; k < 3 * K; k += 2) { const uint2 r = ld_cg_u32x2(sp + k); raw[k] = r.x; raw[k + 1] = r.y; }
                    } else {
#pragma unroll
                        for (uint32_t k = 0; k < K; k++) {
                            const bool have = K * lane + k < nb;
                            raw[3 * k] = have ? ld_cg_u32(sp + 3 * k) : 0u; raw[3 * k + 1] = have ? ld_cg_u32(sp + 3 * k + 1) : 0u; raw[3 * k + 2] = have ? ld_cg_u32(sp + 3 * k + 2) : 1u;
                        }
                    }
                    // prefix form -> lengths: my first record's predecessor is the last record of the lane below (or the carry)
                    uint32_t p_out = __shfl_up_sync(0xffffffffu, raw[3 * (K - 1)], 1), p_lit = __shfl_up_sync(0xffffffffu, raw[3 * (K - 1) + 1], 1);
                    if (lane == 0) { p_out = carry_out; p_lit = carry_lit; }
#pragma unroll
                    for (uint32_t k = 0; k < K; k++) {
                        on[k] = K * lane + k < nb;
                        const uint32_t ll = raw[3 * k + 1] - p_lit, ml = raw[3 * k] - p_out - ll;
                        lls[k] = on[k] ? ll : 0u; mls[k] = on[k] ? ml : 0u; ofs[k] = raw[3 * k + 2];
                        p_out = raw[3 * k]; p_lit = raw[3 * k + 1];
                        pe_out[k] = p_out; pe_lit[k] = p_lit;
                    }
                    {   // carry: the batch's last record
                        const uint32_t lastl = (nb - 1) / K, lasts = (nb - 1) % K;
                        uint32_t co = raw[0], cl = raw[1];
#pragma unroll
                        for (uint32_t k = 1; k < K; k++) { co = lasts == k ? raw[3 * k] : co; cl = lasts == k ? raw[3 * k + 1] : cl; }
                        carry_out = __shfl_sync(0xffffffffu, co, lastl); carry_lit = __shfl_sync(0xffffffffu, cl, lastl);
                    }
                    if (base + EXEC_BATCH < nseq_u && lane * 128u < (nseq_u - base - EXEC_BATCH) * 12u && lane * 128u < EXEC_BATCH * 12u)
                        prefetch_l2(reinterpret_cast<const uint8_t *>(seqs + (uint64_t)(base + EXEC_BATCH) * 3) + lane * 128u);
                }
                // the records are prefix sums already (k_fse): batch totals and batch-relative positions are differences
                const uint32_t T = carry_out - old_out, L = carry_lit - old_lit;
                // per sequence: inclusive end of its bytes, start of its match, inclusive end of its literals (all batch-relative)
                uint32_t oend[K], mstart[K], lend[K];
#pragma unroll
                for (uint32_t k = 0; k < K; k++) { oend[k] = on[k] ? pe_out[k] - old_out : T; lend[k] = on[k] ? pe_lit[k] - old_lit : L; mstart[k] = oend[k] - mls[k]; }
                // actual offsets: symbols resolve against the history at the block's start; a block flagged AUX_RAW_OFFSETS
                // (exact path of k_fse) runs do_offset_history here, sequence by sequence
                uint32_t offs[K];
#pragma unroll
                for (uint32_t k = 0; k < K; k++) offs[k] = resolved ? seq_sym_resolve(ofs[k], bh0, bh1, bh2) : ofs[k];
                uint32_t h0 = st.h0, h1 = st.h1, h2 = st.h2;
                if (!resolved) {
                    // cheap scalar steps (sequence_execution.rs:59-118); committed only if the fast path is taken (the exact path
                    // redoes the steps itself)
                    for (uint32_t j = 0; j < nb; j++) {
                        const uint32_t slot = j % K, src_lane = j / K;
                        uint32_t ll = __shfl_sync(0xffffffffu, exec_pick(lls, slot), src_lane), of = __shfl_sync(0xffffffffu, exec_pick(ofs, slot), src_lane);
                        uint32_t actual = offset_history_step(of, ll, h0, h1, h2);
                        if (lane == src_lane) {
#pragma unroll
                            for (uint32_t k = 0; k < K; k++) offs[k] = slot == k ? actual : offs[k];
                        }
                    }
                }
                const uint64_t reach = st.produced - st.drained;   // bytes of earlier output a match may reach back into
                bool ok = true, ovl = false;
#pragma unroll
                for (uint32_t k = 0; k < K; k++) {
                    ok = ok && (!on[k] || (offs[k] != 0 && (uint64_t)offs[k] <= reach + mstart[k]));
                    ovl = ovl || offs[k] < mls[k];
                }
                const bool fast = __all_sync(0xffffffffu, ok) && T <= EXEC_TMAX && (uint64_t)st.litpos + L <= lit.regen && st.produced + T <= st.cap && !lit.rle;
                if (!fast) {
                    e = exec_batch_exact(st, lit, fd, out, nb, lls, mls, resolved ? offs : ofs, resolved, lane);
                    continue;
                }
                if (!resolved) { st.h0 = h0; st.h1 = h1; st.h2 = h2; }
                // ---------------- fast path
                // Sequence j owns the bytes [lit_begin_j, out_end_j): its literal run, then its match.  A bit is set at
                // the last byte of every sequence, so the owner of output byte q is the number of set bits below q;
                // one 8-byte shared-memory record per sequence then tells the byte where it comes from.
                const uint32_t nrows = (T + 31) >> 5;
                // The batch's match sources are scattered over the frame's window, and with thousands of frames in flight the
                // windows do not stay in L2: ask for the sectors now, a few hundred instructions before the rows need them.
                if (B200Z_EXEC_PREFETCH) {
#pragma unroll
                    for (uint32_t k = 0; k < K; k++) {
                        if (on[k]) {
                            const uint8_t *src = out + st.produced + mstart[k] - offs[k];
                            prefetch_l2(src);
                            if ((((uint32_t)(uintptr_t)src) & 31u) + mls[k] > 32u) prefetch_l2(src + mls[k] - 1);
                        }
                    }
                    if (lane == 31 && lit.regen) {
                        const uint32_t ahead = st.litpos + L + 256u;   // the literal stream is sequential: stay two lines ahead
                        prefetch_l2(lit.p + (ahead < lit.regen ? ahead : lit.regen - 1));
                    }
                }
                sts32(a_mask + (lane << 2), 0u);
                if (nrows > 32u - EXEC_CHUNK_ROWS)
                    for (uint32_t w = lane + 32; w < ((nrows + EXEC_CHUNK_ROWS - 1u) & ~(EXEC_CHUNK_ROWS - 1u)); w += 32) sts32(a_mask + (w << 2), 0u);
                // 8-byte record: literal byte q of the sequence is literal number (q - m_before) of the batch (m_before = match bytes
                // of the earlier sequences = match start - literal end), match byte q comes from output position q - offset
                // (m_start, m_before <= EXEC_TMAX: 16 bits each)
#pragma unroll
                for (uint32_t k = 0; k < K; k += 2)
                    sts128(a_recs + ((K * lane + k) << 3), mstart[k] | ((mstart[k] - lend[k]) << 16), offs[k], mstart[k + 1] | ((mstart[k + 1] - lend[k + 1]) << 16), offs[k + 1]);
                const bool has_ovl = __any_sync(0xffffffffu, ovl);   // some match overlaps its own output (rare)
                __syncwarp();
#pragma unroll
                for (uint32_t k = 0; k < K; k++)
                    if (on[k]) red_or_shared(a_mask + (((oend[k] - 1) >> 5) << 2), 1u << ((oend[k] - 1) & 31u));
                __syncwarp();
                uint8_t *bout = out + st.produced;
                const uint8_t *litq = lit.p + st.litpos;
                asm volatile("" : "+l"(bout), "+l"(litq));   // keep both bases as single 64-bit registers (one add per access)
                uint32_t before = 0;   // sequences ended in earlier rows
                // Rows are produced EXEC_CHUNK_ROWS at a time: every byte whose source lies before the chunk (literals, and
                // matches reaching back past the chunk start) is loaded first -- EXEC_CHUNK_ROWS independent loads per lane in
                // flight -- then stored; the few bytes whose source lies inside the chunk follow, row by row.  (Issuing the
                // next chunk's loads before this chunk's stores was measured slower: more bytes turn dependent.)
                // The per-byte work is branch-free: one select between the literal and the match source.
                // tag: TAG_NONE = nothing to do, TAG_STORE = value loaded, otherwise the (batch-relative, >= floor) source
                // position of a match byte that had to wait.
                constexpr int32_t TAG_NONE = INT32_MIN, TAG_STORE = INT32_MIN + 1;
                constexpr int R = (int)EXEC_CHUNK_ROWS;
                auto load_chunk = [&](uint32_t r0, int32_t floor, uint32_t (&val)[R], int32_t (&tag)[R]) {
#pragma unroll
                    for (int i = 0; i < R; i++) {
                        const uint32_t q = ((r0 + i) << 5) + lane;
                        const uint32_t word = lds32(a_mask + ((r0 + i) << 2));
                        const uint32_t owner = before + __popc(word & lt);   // sequences that ended below q
                        before += __popc(word);
                        const uint2 rc = lds64(a_recs + ((owner & (EXEC_BATCH - 1u)) << 3));
                        const uint32_t mst = rc.x & 0xffffu;
                        const bool is_match = q >= mst;
                        int32_t sp = (int32_t)q - (int32_t)rc.y;                  // batch-relative source of a match byte
                        if (has_ovl) {                                            // overlapping match: byte k comes from k mod offset
                            const uint32_t kk = q - mst;
                            if (is_match && kk >= rc.y) sp = (int32_t)mst - (int32_t)rc.y + (int32_t)(kk % rc.y);
                        }
                        const bool valid = q < T;
                        const bool dep = is_match && sp >= floor;
                        const int32_t idx = is_match ? sp : (int32_t)(q - (rc.x >> 16));
                        const uint8_t *bp = is_match ? (const uint8_t *)bout : litq;
                        tag[i] = valid ? (dep ? sp : TAG_STORE) : TAG_NONE;
                        val[i] = 0;
                        if (valid && !dep) val[i] = bp[idx];
                    }
                };
                auto store_chunk = [&](uint32_t r0, int32_t floor, const uint32_t (&val)[R], const int32_t (&tag)[R]) {
#pragma unroll
                    for (int i = 0; i < R; i++)
                        if (tag[i] == TAG_STORE) bout[((r0 + i) << 5) + lane] = (uint8_t)val[i];
                    // dependent bytes, rows in order (sources in earlier rows are final, inside the row the lowest pending byte is ready)
                    bool anydep = false;
#pragma unroll
                    for (int i = 0; i < R; i++) anydep |= tag[i] >= floor;
                    if (__any_sync(0xffffffffu, anydep)) {
#pragma unroll
                        for (int i = 0; i < R; i++) {
                            bool mine = tag[i] >= floor;
                            uint32_t pending = __ballot_sync(0xffffffffu, mine);
                            const int32_t row0 = (int32_t)((r0 + i) << 5);
                            while (pending) {
                                __syncwarp();
                                bool ready = mine && (tag[i] < row0 || !((pending >> (tag[i] - row0)) & 1u));
                                if (ready) { bout[row0 + (int32_t)lane] = bout[tag[i]]; mine = false; }
                                pending &= ~__ballot_sync(0xffffffffu, ready);
                            }
                        }
                    }
                    __syncwarp();
                };
                for (uint32_t r0 = 0; r0 < nrows; r0 += R) {
                    uint32_t va[R]; int32_t ta[R];
                    load_chunk(r0, (int32_t)(r0 << 5), va, ta);
                    store_chunk(r0, (int32_t)(r0 << 5), va, ta);
                }
                __syncwarp();
                st.produced += T; st.counter += T; st.litpos += L;
            }
            if (!e && st.litpos < lit.regen) {
                uint32_t rest = lit.regen - st.litpos;
                if (st.produced + rest > st.cap) e = B200Z_ERR_TARGET_TOO_SMALL;
                else {
                    if (lit.rle) warp_fill(out + st.produced, lit.byte, rest, lane); else warp_copy(out + st.produced, lit.p + st.litpos, rest, lane);
                    st.produced += rest; st.counter += rest;
                }
            }
            if (!known && !redo && e != B200Z_ERR_CUDA) {
                // everything was consumed (or an execution error came up) before the sequence stage's verdict: it decides
                if (!exec_wait_ready(aux, b, lane)) e = B200Z_ERR_CUDA;
                else {
                    known = true;
                    ax_pad = ld_cg_u32(&aux[b].pad); ax_flags = ld_cg_u32(&aux[b].flags);
                    if (ax_pad) redo = 1; else if (ax_flags & AUX_RAW_OFFSETS) redo = 2;
                }
            }
            if (redo == 2) { redo = 0; goto exec_block_again; }
            if (redo == 1) {   // decode_sequences failed: the reference executes nothing of this block (block_decoder.rs:176-183)
                st = s_saved[threadIdx.x >> 5];
                status = ax_pad; err_block = d.block_in_frame; break;
            }
            if (e) { status = mk_status(e, e == B200Z_ERR_CUDA ? B200Z_STAGE_SEQUENCES : (e == B200Z_ERR_TARGET_TOO_SMALL ? B200Z_STAGE_DRAIN : B200Z_STAGE_EXECUTE)); err_block = d.block_in_frame; break; }
            if (resolved && d.nseq) {   // the history after the block, in terms of the history at its start
                const uint32_t a0 = ld_cg_u32(&aux[b].hist_after[0]), a1 = ld_cg_u32(&aux[b].hist_after[1]), a2 = ld_cg_u32(&aux[b].hist_after[2]);
                st.h0 = seq_sym_resolve(a0, bh0, bh1, bh2); st.h1 = seq_sym_resolve(a1, bh0, bh1, bh2); st.h2 = seq_sym_resolve(a2, bh0, bh1, bh2);
            }
        }
        __syncwarp();
        blocks_done++;
    }
    if (!status && fd.host_status) { status = fd.host_status & 0x00ffffffu; err_block = blocks_done; }
    if (lane == 0) {
        FrameState &o = states[f];
        o.hist[0] = st.h0; o.hist[1] = st.h1; o.hist[2] = st.h2;
        o.status = status; o.produced = st.produced; o.counter = st.counter; o.error_block = err_block; o.blocks_done = blocks_done;
        if (resume) resume[f] = RESUME_SKIP;   // a later launch of this kernel in the same pass has nothing to do here
#ifdef B200Z_PROBE
        { const unsigned long long t = probe_now(); atomicMax(&g_probe[3], t); atomicMin(&g_probe[5], t); }
#endif
    }
}

// ------------------------------------------------------------------------------------------------------------
// k_xxh64: content checksum of every frame's plaintext, XXH64 seed 0 -- what DecodeBuffer feeds on drain
// (decode_buffer.rs:42,225-226,290,301) and FrameDecoder::get_calculated_checksum truncates to 32 bits
// (frame_decoder.rs:262-270).  The four accumulators of XXH64 are independent chains over every 4th 8-byte word:
// four lanes per frame (8 frames per warp), each lane walks its own lane of the 32-byte stripes; lane 0 of the
// group merges and finishes the tail.  Optional stage (B200Z_FLAG_CHECKSUM): it re-reads the output once.
// ------------------------------------------------------------------------------------------------------------
__global__ void k_xxh64(const FrameDesc *__restrict__ frames, FrameState *__restrict__ states, const uint8_t *__restrict__ output, uint32_t nframes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t f = t >> 2, k = t & 3;
    if (f >= nframes) return;
    const FrameState &st = states[f];
    const uint8_t *p = output + frames[f].out_off + st.drained;
    const uint64_t len = st.status ? 0 : st.produced - st.drained;
    const uint64_t h = xxh64_group4(p, len, k);
    if (k == 0) states[f].xxh64 = h;
}

// ------------------------------------------------------------------------------------------------------------
// k_walk: the frame / block / section header walk on the device, for input that lives in device memory (SURVEY 8(f) rank 3,
// first step).  One thread per frame follows the chain of 3-byte block headers (read_block_header, block_decoder.rs:201-283),
// locates the literals and sequences section headers (literals_section.rs:117-223 gives the sizes that locate
// sequence_section.rs:108-167) and hands the host planner exactly the bytes it parses: ~16 bytes per block instead of the whole
// compressed input.  fill == 0: count the blocks; fill == 1: write the digests at first_block[frame].
// ------------------------------------------------------------------------------------------------------------
__global__ void k_walk(const uint8_t *__restrict__ input, uint64_t input_len, const uint64_t *__restrict__ src_off, const uint64_t *__restrict__ src_size,
                       uint32_t nframes, WalkFrame *__restrict__ wf, const uint32_t *__restrict__ first_block, WalkBlock *__restrict__ wb, int fill) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    WalkFrame F;
    for (int i = 0; i < 20; i++) F.hdr[i] = 0;
    F.hdr_avail = 0; F.nblocks = 0; F.stop = 4; F.tail_avail = 0; F.pad = 0; F.end_pos = 0;
    for (int i = 0; i < 4; i++) F.tail[i] = 0;
    const uint64_t so = src_off[f], len = src_size[f];
    if (so <= input_len && len <= input_len - so) {
        const uint8_t *p = input + so;
        F.hdr_avail = (uint32_t)(len < 20 ? len : 20);
        for (uint32_t i = 0; i < F.hdr_avail; i++) F.hdr[i] = p[i];
        // frame header size (frame.rs:6-85); anything wrong with it is the planner's to report
        uint64_t pos = 0;
        bool ok = len >= 5 && (uint32_t)(F.hdr[0] | (F.hdr[1] << 8) | (F.hdr[2] << 16) | ((uint32_t)F.hdr[3] << 24)) == 0xFD2FB528u;
        if (ok) {
            const uint32_t desc = F.hdr[4], single = (desc >> 5) & 1u, flag = desc >> 6;
            const uint32_t dl = (desc & 3u) == 3u ? 4u : (desc & 3u);
            const uint32_t fl = flag == 0 ? single : (flag == 1 ? 2u : (flag == 2 ? 4u : 8u));
            pos = 5u + (single ? 0u : 1u) + dl + fl;
            ok = len >= pos;
        }
        if (ok) {
            uint32_t nb = 0;
            const uint32_t base = fill ? first_block[f] : 0u;
            for (;;) {
                if (len - pos < 3) { F.stop = 1; break; }
                const uint32_t b0 = p[pos], b1 = p[pos + 1], b2 = p[pos + 2];
                const uint32_t t = (b0 >> 1) & 3u, size = (b0 >> 3) | (b1 << 5) | (b2 << 13);
                WalkBlock B;
                B.pos = pos; B.seq_off = 0; B.bh[0] = (uint8_t)b0; B.bh[1] = (uint8_t)b1; B.bh[2] = (uint8_t)b2; B.lit_avail = 0; B.seq_avail = 0;
                for (int i = 0; i < 5; i++) B.lit[i] = 0;
                for (int i = 0; i < 4; i++) B.seq[i] = 0;
                for (int i = 0; i < 6; i++) B.pad[i] = 0;
                if (t == 3 || size > 128u * 1024u) {   // the planner reports FoundReservedBlock / BlockSizeTooLarge from these 3 bytes
                    if (fill) wb[base + nb] = B;
                    nb++; F.stop = 2; break;
                }
                const uint32_t content = t == BT_RLE ? 1u : size;
                pos += 3;
                if (len - pos < content) {
                    if (fill) wb[base + nb] = B;
                    nb++; F.stop = 3; break;
                }
                if (t == BT_COMPRESSED && size) {
                    const uint8_t *c = p + pos;
                    B.lit_avail = (uint8_t)(size < 5 ? size : 5);
                    for (uint32_t i = 0; i < B.lit_avail; i++) B.lit[i] = c[i];
                    const uint32_t lt = c[0] & 3u, sf = (c[0] >> 2) & 3u;
                    const uint32_t need = (lt == LT_RAW || lt == LT_RLE) ? ((sf == 0 || sf == 2) ? 1u : (sf == 1 ? 2u : 3u)) : (sf <= 1 ? 3u : (sf == 2 ? 4u : 5u));
                    if (size >= need) {
                        uint32_t regen, comp = 0;
                        if (lt == LT_RAW || lt == LT_RLE) {
                            if (sf == 0 || sf == 2) regen = c[0] >> 3;
                            else if (sf == 1) regen = (c[0] >> 4) + ((uint32_t)c[1] << 4);
                            else regen = (c[0] >> 4) + ((uint32_t)c[1] << 4) + ((uint32_t)c[2] << 12);
                        } else if (sf <= 1) { regen = (c[0] >> 4) + (((uint32_t)c[1] & 0x3f) << 4); comp = (c[1] >> 6) + ((uint32_t)c[2] << 2); }
                        else if (sf == 2) { regen = (c[0] >> 4) + ((uint32_t)c[1] << 4) + (((uint32_t)c[2] & 3) << 12); comp = (c[2] >> 2) + ((uint32_t)c[3] << 6); }
                        else { regen = (c[0] >> 4) + ((uint32_t)c[1] << 4) + (((uint32_t)c[2] & 0x3f) << 12); comp = (c[2] >> 6) + ((uint32_t)c[3] << 2) + ((uint32_t)c[4] << 10); }
                        const uint32_t upper = (lt == LT_COMPRESSED || lt == LT_TREELESS) ? comp : (lt == LT_RLE ? 1u : regen);
                        if (size - need >= upper) {
                            const uint32_t rem = size - need - upper;
                            B.seq_off = need + upper;
                            B.seq_avail = (uint8_t)(rem < 4 ? rem : 4);
                            for (uint32_t i = 0; i < B.seq_avail; i++) B.seq[i] = c[need + upper + i];
                        }
                    }
                }
                if (fill) wb[base + nb] = B;
                nb++;
                pos += content;
                if (b0 & 1u) {   // last block: the content checksum may follow
                    F.stop = 0;
                    const uint64_t left = len - pos;
                    F.tail_avail = (uint32_t)(left < 4 ? left : 4);
                    for (uint32_t i = 0; i < F.tail_avail; i++) F.tail[i] = p[pos + i];
                    break;
                }
            }
            F.nblocks = nb; F.end_pos = pos;
        }
    }
    wf[f] = F;
}

}  // namespace b200z

#include "fse2.cuh"
#include "exec_cta.cuh"

namespace b200z {

// ------------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------------
static inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

int launch_predefined(FseSlot *predef, cudaStream_t s) {
    k_predefined<<<1, 32, 0, s>>>(predef);
    return (int)cudaGetLastError();
}

constexpr uint32_t kHufSmem = HUF_BLOCKS_PER_CTA * HUF_SMEM_PER_BLOCK + 32 * RING_STRIDE;
constexpr uint32_t kFseSmem = FSE_BLOCKS_PER_CTA * FSE_TAB_U16 * 2 + 1024 + FSE_BLOCKS_PER_CTA * RING_STRIDE;

static int g_num_sms[64];   // per device ordinal, filled by init_kernels

int init_kernels() {
    cudaError_t e = cudaFuncSetAttribute(k_fse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFseSmem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_huf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHufSmem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_fse2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFse2Smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_fse2, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_exec_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XC_SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    // k_fse and k_huf run side by side: ask for the largest shared-memory carve-out so that both fit
    e = cudaFuncSetAttribute(k_fse, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_huf, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    int dev = 0, sms = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    if (dev >= 0 && dev < 64) g_num_sms[dev] = sms;
    return 0;
}

uint32_t num_sms() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || g_num_sms[dev] <= 0) return 148;
    return (uint32_t)g_num_sms[dev];
}

const char *const kStageNames[kNumStages] = {"k_setup", "k_huf", "k_fse", "k_exec_cta", "k_exec"};

// one stage of the pipeline; a stage with nothing to do launches nothing and returns 0
int launch_stage(const PipelineArgs &a, int stage, cudaStream_t s) {
    switch (stage) {
        case 0: if (a.nblocks) k_setup<<<cdiv(a.nblocks, SETUP_WARPS), SETUP_WARPS * 32, 0, s>>>(a.descs, a.aux, a.input, a.nblocks, 3u); break;
        case 1:
            if (a.nblocks)
                k_huf<<<cdiv(a.nblocks, HUF_BLOCKS_PER_CTA), 32, kHufSmem, s>>>(a.descs, a.aux, a.input, a.lit_scratch, a.nblocks);
            break;
        case 2:
            if (a.nblocks) {
                // default: one warp walks chain and values (106 instructions per sequence).  B200Z_FSE=2: chain warp + value warp
                // through a shared-memory queue (k_fse2) -- measured slower on B200 (1.34 vs 1.13 ms on C2b: the chain only drops to
                // 92 instructions and pays for the queue hand-off), kept for A/B runs.
                static const bool one_warp = [] { const char *e = getenv("B200Z_FSE"); return !(e && e[0] == '2'); }();
                if (one_warp) k_fse<<<cdiv(a.nblocks, FSE_BLOCKS_PER_CTA), 32, kFseSmem, s>>>(a.descs, a.aux, a.input, a.seq_scratch, a.nblocks, a.fse_order);
                else k_fse2<<<cdiv(a.nblocks, F2_LANES), 64, kFse2Smem, s>>>(a.descs, a.aux, a.input, a.seq_scratch, a.nblocks);
            }
            break;
        case 3:
            // frames whose blocks are assembled in shared memory: persistent CTAs, one per SM, frames from a ticket counter
            if (a.nframes && a.n_cta_frames)
                k_exec_cta<<<a.n_cta_frames < num_sms() ? a.n_cta_frames : num_sms(), XC_THREADS, XC_SMEM_BYTES, s>>>(
                    a.descs, a.aux, a.frames, a.states, a.input, a.lit_scratch, a.seq_scratch, a.output, a.output_cap, a.cta_frames, a.n_cta_frames, a.resume,
                    a.ticket);
            break;
        case 4:
            // every other frame, and whatever k_exec_cta left (resume[]): one warp per frame
            if (a.nframes) {
                // optional waves (B200Z_EXEC_WAVE frames per launch): fewer live windows, so match sources stay in L2
                static const uint32_t wave = [] { const char *e = getenv("B200Z_EXEC_WAVE"); return e ? (uint32_t)strtoul(e, nullptr, 10) : 0u; }();
                const uint32_t step = wave ? wave : a.nframes;
                for (uint32_t base = 0; base < a.nframes; base += step) {
                    const uint32_t n = a.nframes - base < step ? a.nframes - base : step;
                    k_exec<<<cdiv(n, EXEC_WARPS), EXEC_WARPS * 32, 0, s>>>(a.descs, a.aux, a.frames, a.states, a.input, a.lit_scratch, a.seq_scratch,
                                                                 a.output, a.output_cap, base + n, a.resume, base);
                }
            }
            break;
        default: break;
    }
    return (int)cudaGetLastError();
}

int launch_walk(const uint8_t *d_input, uint64_t input_len, const uint64_t *d_src_off, const uint64_t *d_src_size, uint32_t nframes, WalkFrame *d_wf,
                const uint32_t *d_first_block, WalkBlock *d_wb, int fill, cudaStream_t s) {
    if (nframes) k_walk<<<cdiv(nframes, 128), 128, 0, s>>>(d_input, input_len, d_src_off, d_src_size, nframes, d_wf, d_first_block, d_wb, fill);
    return (int)cudaGetLastError();
}

int launch_checksum(const PipelineArgs &a, cudaStream_t s) {
    if (a.nframes) k_xxh64<<<cdiv(a.nframes * 4, 128), 128, 0, s>>>(a.frames, a.states, a.output, a.nframes);
    return (int)cudaGetLastError();
}

// resume[] and the ticket counter start from their initial image for every pass
int reset_sched(const PipelineArgs &a, cudaStream_t s) {
    if (!a.nframes || !a.ticket) return 0;
    return (int)cudaMemcpyAsync(a.ticket, a.sched_init, a.sched_bytes, cudaMemcpyDeviceToDevice, s);
}

int launch_pipeline(const PipelineArgs &a, cudaStream_t s) {
    if (int e = reset_sched(a, s)) return e;
    for (int st = 0; st < kNumStages; st++) { int e = launch_stage(a, st, s); if (e) return e; }
    return 0;
}

static int launch_exec_warp(const PipelineArgs &a, cudaStream_t s, bool dependent_of_fse) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cdiv(a.nframes, EXEC_WARPS)); cfg.blockDim = dim3(EXEC_WARPS * 32); cfg.dynamicSmemBytes = 0; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    static const bool no_pdl = [] { const char *e = getenv("B200Z_EXEC_PDL"); return e && e[0] == '0'; }();   // A/B knob: k_exec strictly after k_fse
    cfg.attrs = attr; cfg.numAttrs = dependent_of_fse && !no_pdl ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, k_exec, a.descs, (const BlockAux *)a.aux, a.frames, a.states, a.input, (const uint8_t *)a.lit_scratch,
                                   (const uint32_t *)a.seq_scratch, a.output, a.output_cap, a.nframes, a.resume, 0u);
}

// The shipped launch order.  k_exec (one warp per frame) runs BESIDE k_fse: it is launched in the same stream as k_fse's
// programmatic dependent (every k_fse CTA executes griddepcontrol.launch_dependents first thing, so all of them are resident
// before the first k_exec CTA takes an SM; k_exec never calls griddepcontrol.wait) and starts a frame's block as soon as that
// block's sequence stage is over (BlockAux::ready).  k_fse is a latency-bound chain that leaves most issue slots idle; k_exec is
// issue-bound.  Frames of k_exec_cta follow when k_fse is complete, then k_exec once more for whatever k_exec_cta handed back.
// (k_huf beside k_fse on a second stream was measured: no gain -- both want the shared memory of every SM.)
int launch_pipeline_overlapped(const PipelineArgs &a, const PipelineStreams &ps) {
    int e;
    if ((e = reset_sched(a, ps.main))) return e;
    if ((e = launch_tables_literals(a, ps))) return e;
    if ((e = launch_fse_exec(a, ps.main))) return e;
    return launch_cta_rest(a, ps.main);
}

// k_setup (both sides) and k_huf
int launch_tables_literals(const PipelineArgs &a, const PipelineStreams &ps) {
    int e;
    if (a.nblocks && ps.side && ps.fork && ps.join) {
        // literals side (Huffman tables, then k_huf) on the side stream, beside the FSE table builds on the main stream; both are
        // done before k_fse starts, so that k_exec stays k_fse's immediate successor
        if ((e = (int)cudaEventRecord(ps.fork, ps.main))) return e;
        if ((e = (int)cudaStreamWaitEvent(ps.side, ps.fork, 0))) return e;
        k_setup<<<cdiv(a.nblocks, SETUP_WARPS), SETUP_WARPS * 32, 0, ps.side>>>(a.descs, a.aux, a.input, a.nblocks, 1u);
        if ((e = (int)cudaGetLastError())) return e;
        if ((e = launch_stage(a, 1, ps.side))) return e;
        if ((e = (int)cudaEventRecord(ps.join, ps.side))) return e;
        k_setup<<<cdiv(a.nblocks, SETUP_WARPS), SETUP_WARPS * 32, 0, ps.main>>>(a.descs, a.aux, a.input, a.nblocks, 2u);
        if ((e = (int)cudaGetLastError())) return e;
        if ((e = (int)cudaStreamWaitEvent(ps.main, ps.join, 0))) return e;
    } else {
        if ((e = launch_stage(a, 0, ps.main))) return e;
        if ((e = launch_stage(a, 1, ps.main))) return e;
    }
    return 0;
}

// k_fse and, beside it, k_exec for the frames of the warp kernel
int launch_fse_exec(const PipelineArgs &a, cudaStream_t s) {
    int e;
    if ((e = launch_stage(a, 2, s))) return e;
    if (!a.nframes || a.n_cta_frames >= a.nframes) return 0;
    return launch_exec_warp(a, s, a.nblocks != 0);
}

// k_exec_cta for its frames, then k_exec for what it handed back
int launch_cta_rest(const PipelineArgs &a, cudaStream_t s) {
    if (!a.nframes || !a.n_cta_frames) return 0;
    if (int e = launch_stage(a, 3, s)) return e;
    return launch_exec_warp(a, s, false);
}

// launches of launch_pipeline_overlapped
uint32_t pipeline_launch_count(const PipelineArgs &a) {
    return (a.nblocks ? 4u : 0u) + (a.nframes && a.n_cta_frames < a.nframes ? 1u : 0u) + (a.nframes && a.n_cta_frames ? 2u : 0u);
}

}  // namespace b200z
