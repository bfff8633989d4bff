// compress.cu -- batch zstd frame compression (ruzstd encoding::FrameCompressor at CompressionLevel::{Uncompressed, Fastest},
// frame_compressor.rs:131-224, levels/fastest.rs:20-69).  A 128 KiB block is the unit of work: the Fastest matcher never
// looks outside the current block (MatchGeneratorDriver::new(128 KiB, 1), match_generator.rs:28-53), so every block of every
// frame is compressed at once.  Kernels, in launch order (DESIGN.md section 9):
//   k_cxxh64  content checksum of every frame's plaintext (xxh64.cuh, shared with k_xxh64)
//   k_cmatch  one CTA per block: all-equal test (RLE block), hash-table candidates, greedy parse by segments -> sequences and
//             literals in the block's scratch
//   k_cblock  one warp per block: histograms, Huffman / FSE tables and their descriptions (lane 0/1), the four Huffman streams
//             (lanes 0..3) and the sequences stream (lane 4); Raw when the result is not smaller than the block
//   k_cframe  one warp per frame: prefix sum of block sizes, frame header, checksum, TARGET_TOO_SMALL
//   k_cemit   block headers and bodies at their final place
// Every output byte is a function of the frame's plaintext, the level and the flags: the only atomics are histogram counts
// and atomicMax on hash-table positions.
#include <cub/block/block_scan.cuh>
#include <cuda_runtime.h>

#include "compress.h"
#include "enc.cuh"
#include "xxh64.cuh"

namespace b200z {

const char *const kCompressKernelNames[kCompressKernels] = {"k_cxxh64", "k_cmatch", "k_cblock", "k_cframe", "k_cemit"};

// ---- k_cxxh64 -------------------------------------------------------------------------------------------------------------
__global__ void k_cxxh64(const CFrame *__restrict__ frames, const uint8_t *__restrict__ input, uint64_t *__restrict__ hash, uint32_t nframes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t f = t >> 2, k = t & 3;
    if (f >= nframes) return;
    const uint64_t h = xxh64_group4(input + frames[f].src_off, frames[f].src_size, k);
    if (k == 0) hash[f] = h;
}

// ---- k_cmatch -------------------------------------------------------------------------------------------------------------
constexpr uint32_t CM_THREADS = 256;
constexpr uint32_t CM_SEG = ENC_BLOCK / CM_THREADS;   // bytes parsed by one thread; matches are clipped at its end
constexpr uint32_t CM_HASH_LOG = 13;
constexpr uint32_t CM_SMEM = ENC_BLOCK + 16 + (4u << CM_HASH_LOG);
static_assert(ENC_MAX_SEQ >= CM_THREADS * (CM_SEG / ENC_MIN_MATCH), "sequence scratch too small for k_cmatch's segments");

__device__ __forceinline__ uint32_t cm_hash(const uint8_t *d, uint32_t p) {
    const uint32_t v = (uint32_t)d[p] | ((uint32_t)d[p + 1] << 8) | ((uint32_t)d[p + 2] << 16) | ((uint32_t)d[p + 3] << 24);
    return (v * 2654435761u) >> (32 - CM_HASH_LOG);
}

// Greedy parse of [s0, s1): a candidate is taken when it matches for ENC_MIN_MATCH bytes or more; the match is extended up to
// s1.  `prev_end` = where the previous match of the block ended (the first sequence's literal length counts from there).
template <bool WRITE>
__device__ void cm_parse(const uint8_t *d, const uint32_t *cand, uint32_t s0, uint32_t s1, uint32_t prev_end, EncSeq *seqs, uint8_t *lits,
                         uint32_t &nseq, uint32_t &nlit, int32_t &last_end) {
    uint32_t p = s0, anchor = s0;
    nseq = 0; nlit = 0; last_end = -1;
    while (p + ENC_MIN_MATCH <= s1) {
        const uint32_t c = cand[p];
        uint32_t len = 0;
        if (c) {
            const uint32_t q = c - 1, maxlen = s1 - p;
            while (len < maxlen && d[q + len] == d[p + len]) len++;
        }
        if (len >= ENC_MIN_MATCH) {
            if (WRITE) {
                for (uint32_t i = anchor; i < p; i++) lits[nlit + i - anchor] = d[i];
                seqs[nseq] = EncSeq{p - prev_end, len, p - (c - 1)};
            }
            nlit += p - anchor;
            nseq++;
            p += len;
            anchor = prev_end = p;
            last_end = (int32_t)p;
        } else p++;
    }
    if (WRITE) for (uint32_t i = anchor; i < s1; i++) lits[nlit + i - anchor] = d[i];
    nlit += s1 - anchor;
}

__global__ void __launch_bounds__(CM_THREADS) k_cmatch(const CBlock *__restrict__ blocks, CBlockOut *__restrict__ bout, const uint8_t *__restrict__ input,
                                                       uint32_t *__restrict__ cand_all, uint8_t *__restrict__ lits_all, EncSeq *__restrict__ seqs_all,
                                                       uint32_t nblocks) {
    extern __shared__ __align__(16) uint8_t sm[];
    uint8_t *d = sm;
    uint32_t *ht = reinterpret_cast<uint32_t *>(sm + ENC_BLOCK + 16);
    __shared__ int32_t last_end_s[CM_THREADS];
    using Scan = cub::BlockScan<unsigned long long, CM_THREADS>;
    __shared__ typename Scan::TempStorage scan_tmp;
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    uint32_t *cand = cand_all + (size_t)blockIdx.x * ENC_BLOCK;
    for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const CBlock blk = blocks[b];
        const uint32_t n = blk.n;
        const uint8_t *src = input + blk.src_off;
        for (uint32_t i = tid; i < n; i += CM_THREADS) d[i] = src[i];
        if (tid < 16) d[n + tid] = 0;
        for (uint32_t i = tid; i < (1u << CM_HASH_LOG); i += CM_THREADS) ht[i] = 0;
        __syncthreads();
        bool same = true;
        for (uint32_t i = tid; i < n; i += CM_THREADS) same &= d[i] == d[0];
        same = __syncthreads_and(same);
        if (n == 0 || same) {
            if (tid == 0) bout[b] = CBlockOut{n ? BT_RLE : BT_RAW, n ? 1u : 0u, 0, 0};
            __syncthreads();
            continue;
        }
        // candidates in position order, blockDim positions at a time: look up (the most recent earlier position of the same hash
        // in an earlier chunk, or the nearest earlier lane of this warp with the same hash), then insert with atomicMax
        for (uint32_t base = 0; base < n; base += CM_THREADS) {
            const uint32_t p = base + tid;
            const bool valid = p + ENC_MIN_MATCH <= n;
            const uint32_t h = valid ? cm_hash(d, p) : (0x80000000u | tid);
            const uint32_t same_h = __match_any_sync(0xffffffffu, h) & ((1u << lane) - 1u);
            if (p < n) cand[p] = !valid ? 0u : (same_h ? p - lane + (31u - __clz(same_h)) + 1u : ht[h]);
            __syncthreads();
            if (valid) atomicMax(&ht[h], p + 1);
            __syncthreads();
        }
        // greedy parse by segments: count, place by a prefix sum, parse again writing
        const uint32_t s0 = min(n, tid * CM_SEG), s1 = min(n, s0 + CM_SEG);
        uint32_t ns, nl;
        int32_t le;
        cm_parse<false>(d, cand, s0, s1, 0, nullptr, nullptr, ns, nl, le);
        last_end_s[tid] = le;
        unsigned long long pre, tot;
        Scan(scan_tmp).ExclusiveSum(((unsigned long long)ns << 32) | nl, pre, tot);
        __syncthreads();
        uint32_t prev_end = 0;
        for (int32_t t = (int32_t)tid - 1; t >= 0; t--) if (last_end_s[t] >= 0) { prev_end = (uint32_t)last_end_s[t]; break; }
        cm_parse<true>(d, cand, s0, s1, prev_end, seqs_all + (size_t)b * ENC_MAX_SEQ + (pre >> 32), lits_all + (size_t)b * ENC_BLOCK + (uint32_t)pre,
                       ns, nl, le);
        if (tid == 0) bout[b] = CBlockOut{BT_COMPRESSED, 0, (uint32_t)(tot >> 32), (uint32_t)tot};
        __syncthreads();
    }
}

// ---- k_cblock -------------------------------------------------------------------------------------------------------------
constexpr uint32_t CB_WARPS = 4;
struct CBlockSmem {
    LitPlan L;
    SeqPlan S;
    uint32_t hist[256], hll[36], hof[32], hml[53];
    uint8_t spread[512];
    uint32_t lsz, ssz;
};

__global__ void __launch_bounds__(CB_WARPS * 32) k_cblock(const CBlock *__restrict__ blocks, CBlockOut *__restrict__ bout, const uint8_t *__restrict__ input,
                                                         const uint8_t *__restrict__ lits_all, const EncSeq *__restrict__ seqs_all,
                                                         uint8_t *__restrict__ body_all, uint32_t nblocks) {
    extern __shared__ __align__(16) uint8_t sm[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * CB_WARPS + warp;
    if (b >= nblocks) return;
    CBlockSmem &W = reinterpret_cast<CBlockSmem *>(sm)[warp];
    const CBlockOut o = bout[b];
    if (o.type != BT_COMPRESSED) return;
    const uint32_t n = blocks[b].n, nlit = o.nlit, nseq = o.nseq;
    const uint8_t *lits = lits_all + (size_t)b * ENC_BLOCK;
    const EncSeq *seqs = seqs_all + (size_t)b * ENC_MAX_SEQ;
    uint8_t *body = body_all + (size_t)b * ENC_BODY_STRIDE;
    for (uint32_t i = lane; i < 256; i += 32) W.hist[i] = 0;
    for (uint32_t i = lane; i < 36; i += 32) W.hll[i] = 0;
    W.hof[lane] = 0;
    for (uint32_t i = lane; i < 53; i += 32) W.hml[i] = 0;
    __syncwarp();
    uint32_t xb, xe;
    for (uint32_t i = lane; i < nlit; i += 32) atomicAdd(&W.hist[lits[i]], 1u);
    for (uint32_t i = lane; i < nseq; i += 32) {
        const EncSeq q = seqs[i];
        atomicAdd(&W.hll[enc_ll_code(q.ll, xb, xe)], 1u);
        atomicAdd(&W.hof[enc_of_code(q.off, xb, xe)], 1u);
        atomicAdd(&W.hml[enc_ml_code(q.ml, xb, xe)], 1u);
    }
    __syncwarp();
    if (lane == 0) lit_plan(W.hist, nlit, W.L);
    if (lane == 1) seq_plan(nseq, W.hll, W.hof, W.hml, W.S, W.spread);
    __syncwarp();
    const bool huf = W.L.type == LT_COMPRESSED;
    uint32_t soff = 0, scnt = 0;
    if (huf && lane < 4) {
        huf_stream_split(nlit, lane, soff, scnt);
        W.L.stream_size[lane] = huf_stream_bytes(lits + soff, scnt, W.L.len);
    }
    __syncwarp();
    if (lane == 0) W.lsz = lit_finish(W.L);
    __syncwarp();
    const uint32_t lsz = W.lsz, cap = n;
    if (lsz <= cap) {
        const uint32_t type = W.L.type;
        if (type == LT_RAW) {
            if (lane == 0) for (uint32_t i = 0; i < W.L.hdr_size; i++) body[i] = W.L.hdr[i];
            for (uint32_t i = lane; i < nlit; i += 32) body[W.L.hdr_size + i] = lits[i];
        } else {
            if (lane == 0) lit_write_prefix(body, W.L, lits);
            if (type == LT_COMPRESSED && lane < 4) {
                uint32_t at = W.L.hdr_size + W.L.desc_size + 6;
                for (uint32_t k = 0; k < lane; k++) at += W.L.stream_size[k];
                huf_encode_stream(body + at, W.L.stream_size[lane], lits + soff, scnt, W.L.code, W.L.len);
            }
        }
        if (lane == 4) W.ssz = seq_write(body + lsz, cap - lsz, seqs, W.S);
    }
    __syncwarp();
    if (lane == 0) {
        const uint32_t total = lsz <= cap ? lsz + W.ssz : cap + 1;
        bout[b] = total >= n ? CBlockOut{BT_RAW, n, nseq, nlit} : CBlockOut{BT_COMPRESSED, total, nseq, nlit};
    }
}

// ---- k_cframe -------------------------------------------------------------------------------------------------------------
__global__ void k_cframe(const CFrame *__restrict__ frames, const CBlock *__restrict__ blocks, CBlockOut *__restrict__ bout, uint64_t *__restrict__ block_off,
                         const uint64_t *__restrict__ hash, uint8_t *__restrict__ output, uint64_t output_cap, b200z_compress_result *__restrict__ results,
                         uint32_t nframes, uint32_t level, uint32_t flags) {
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= nframes) return;
    const CFrame F = frames[f];
    uint8_t hdr[16];
    const uint32_t hsz = enc_frame_header(hdr, flags, F.src_size);
    uint64_t run = hsz;
    uint32_t nraw = 0, nrle = 0, ncomp = 0;
    for (uint32_t base = 0; base < F.nblocks; base += 32) {
        const uint32_t b = F.first_block + base + lane;
        uint64_t sz = 0;
        if (base + lane < F.nblocks) {
            if (level == 0) bout[b] = CBlockOut{BT_RAW, blocks[b].n, 0, 0};
            const CBlockOut o = bout[b];
            sz = 3 + o.size;
            nraw += o.type == BT_RAW; nrle += o.type == BT_RLE; ncomp += o.type == BT_COMPRESSED;
        }
        uint64_t incl = sz;
        for (int d = 1; d < 32; d <<= 1) { const uint64_t v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += v; }
        if (base + lane < F.nblocks) block_off[b] = run + incl - sz;
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
    for (int d = 16; d; d >>= 1) {
        nraw += __shfl_xor_sync(0xffffffffu, nraw, d); nrle += __shfl_xor_sync(0xffffffffu, nrle, d); ncomp += __shfl_xor_sync(0xffffffffu, ncomp, d);
    }
    if (lane) return;
    const uint64_t total = run + ((flags & ENC_FLAG_CHECKSUM) ? 4 : 0);
    b200z_compress_result r;
    r.num_blocks = F.nblocks; r.raw_blocks = nraw; r.rle_blocks = nrle; r.compressed_blocks = ncomp;
    r.checksum = (flags & ENC_FLAG_CHECKSUM) ? (uint32_t)hash[f] : 0u;
    r.reserved = 0; r.stage = 0;
    if (total > F.out_cap || F.out_off > output_cap || total > output_cap - F.out_off) {
        r.status = B200Z_ERR_TARGET_TOO_SMALL; r.out_size = 0;
    } else {
        r.status = 0; r.out_size = total;
        uint8_t *o = output + F.out_off;
        for (uint32_t i = 0; i < hsz; i++) o[i] = hdr[i];
        if (flags & ENC_FLAG_CHECKSUM) for (int i = 0; i < 4; i++) o[run + i] = (uint8_t)(r.checksum >> (8 * i));
    }
    results[f] = r;
}

// ---- k_cemit --------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cemit(const CFrame *__restrict__ frames, const CBlock *__restrict__ blocks, const CBlockOut *__restrict__ bout,
                                               const uint64_t *__restrict__ block_off, const b200z_compress_result *__restrict__ results,
                                               const uint8_t *__restrict__ input, const uint8_t *__restrict__ body_all, uint8_t *__restrict__ output,
                                               uint32_t nblocks) {
    for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const CBlock blk = blocks[b];
        if (results[blk.frame].status) continue;
        const CBlockOut o = bout[b];
        uint8_t *dst = output + frames[blk.frame].out_off + block_off[b];
        if (threadIdx.x == 0) enc_block_header(dst, blk.last, o.type, o.type == BT_RLE ? blk.n : o.size);
        dst += 3;
        const uint8_t *src = o.type == BT_COMPRESSED ? body_all + (size_t)b * ENC_BODY_STRIDE : input + blk.src_off;
        const uint32_t len = o.size;
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) dst[i] = src[i];
    }
}

// ---- launch ---------------------------------------------------------------------------------------------------------------
int init_compress_kernels(uint32_t *match_ctas) {
    int dev = 0, sms = 0, per = 0;
    cudaError_t e;
    if ((e = cudaGetDevice(&dev)) || (e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) ||
        (e = cudaFuncSetAttribute(k_cmatch, cudaFuncAttributeMaxDynamicSharedMemorySize, CM_SMEM)) ||
        (e = cudaFuncSetAttribute(k_cblock, cudaFuncAttributeMaxDynamicSharedMemorySize, CB_WARPS * sizeof(CBlockSmem))) ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_cmatch, CM_THREADS, CM_SMEM)))
        return (int)e;
    if (per < 1) return (int)cudaErrorInvalidConfiguration;
    *match_ctas = (uint32_t)(sms * per);
    return 0;
}

int launch_compress_stage(const CompressArgs &a, int stage, cudaStream_t s) {
    if (!a.nframes) return 0;
    switch (stage) {
    case 0: if (a.flags & ENC_FLAG_CHECKSUM) k_cxxh64<<<(a.nframes * 4 + 127) / 128, 128, 0, s>>>(a.frames, a.input, a.hash, a.nframes); break;
    case 1: if (a.level) k_cmatch<<<a.match_ctas < a.nblocks ? a.match_ctas : a.nblocks, CM_THREADS, CM_SMEM, s>>>(a.blocks, a.bout, a.input, a.cand, a.lits, a.seqs, a.nblocks); break;
    case 2: if (a.level) k_cblock<<<(a.nblocks + CB_WARPS - 1) / CB_WARPS, CB_WARPS * 32, CB_WARPS * sizeof(CBlockSmem), s>>>(a.blocks, a.bout, a.input, a.lits, a.seqs, a.body, a.nblocks); break;
    case 3: k_cframe<<<(a.nframes + 3) / 4, 128, 0, s>>>(a.frames, a.blocks, a.bout, a.block_off, a.hash, a.output, a.output_cap, a.results, a.nframes, a.level, a.flags); break;
    case 4: k_cemit<<<a.nblocks < 65535u * 16 ? a.nblocks : 65535u * 16, 256, 0, s>>>(a.frames, a.blocks, a.bout, a.block_off, a.results, a.input, a.body, a.output, a.nblocks); break;
    }
    return (int)cudaGetLastError();
}

uint32_t compress_launch_count(const CompressArgs &a) {
    if (!a.nframes) return 0;
    return 2 + ((a.flags & ENC_FLAG_CHECKSUM) ? 1 : 0) + (a.level ? 2 : 0);
}

}  // namespace b200z
