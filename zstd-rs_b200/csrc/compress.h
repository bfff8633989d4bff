// compress.h -- launch interface between the host library (api.cpp) and the compression kernels (compress.cu)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200zstd.h"
#include "enc.cuh"

namespace b200z {

constexpr uint32_t ENC_MAX_SEQ = (ENC_BLOCK / 256) / ENC_MIN_MATCH * 256;   // k_cmatch: 256 segments, each match >= ENC_MIN_MATCH bytes
constexpr uint32_t ENC_BODY_STRIDE = ENC_BLOCK + 64;                       // a compressed body is kept only if smaller than its block

struct CBlock { uint64_t src_off; uint32_t n, frame, last, pad; };   // one per 128 KiB block (host plan)
struct CBlockOut { uint32_t type, size, nseq, nlit; };               // block type and body size (size 1 for RLE); sequences, literals
struct CFrame { uint64_t src_off, src_size, out_off, out_cap; uint32_t first_block, nblocks; };

struct CompressArgs {
    const uint8_t *input;      // device: plaintext of every frame
    uint8_t *output;           // device
    uint64_t output_cap;
    const CFrame *frames;      // [nframes] device
    const CBlock *blocks;      // [nblocks] device
    CBlockOut *bout;           // [nblocks] device
    uint64_t *block_off;       // [nblocks] device: block header position inside its frame
    uint64_t *hash;            // [nframes] device: XXH64 of each frame's plaintext
    b200z_compress_result *results;   // [nframes] device
    uint8_t *lits;             // [nblocks * ENC_BLOCK] scratch
    EncSeq *seqs;              // [nblocks * ENC_MAX_SEQ] scratch
    uint8_t *body;             // [nblocks * ENC_BODY_STRIDE] scratch
    uint32_t *cand;            // [match_ctas * ENC_BLOCK] scratch: match candidate of every position of the block in flight
    uint32_t nblocks, nframes, level, flags, match_ctas;
};

constexpr int kCompressKernels = 5;
extern const char *const kCompressKernelNames[kCompressKernels];
// per device, at context creation: kernel attributes (k_cmatch's and k_cblock's dynamic shared memory) and the number of k_cmatch
// CTAs resident on the current device at once (sizes the `cand` scratch); a cudaError_t, 0 = ok
int init_compress_kernels(uint32_t *match_ctas);
int launch_compress_stage(const CompressArgs &a, int stage, cudaStream_t s);   // stage < kCompressKernels, in order
uint32_t compress_launch_count(const CompressArgs &a);

}  // namespace b200z
