// api.cpp -- the C ABI declared in include/b200zstd.h: context, dictionaries, batch entry (tier 1) and the
// FrameDecoder / StreamingDecoder mirrors (tier 2).  Host logic only; all decoding happens in kernels.cu.
// There is no CPU decode path in this library: without a usable CUDA device b200z_ctx_create fails.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/b200zstd.h"
#include "compress.h"
#include "kernels.h"
#include "plan.h"
#include "tables.cuh"

using namespace b200z;

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct ErrName { int code; const char *name; };
#define EN(x) {B200Z_##x, #x}
const ErrName kErrNames[] = {
    EN(OK), EN(ERR_MAGIC_NUMBER_READ), EN(ERR_BAD_MAGIC_NUMBER), EN(ERR_FRAME_DESCRIPTOR_READ), EN(ERR_INVALID_FRAME_DESCRIPTOR),
    EN(ERR_WINDOW_DESCRIPTOR_READ), EN(ERR_DICTIONARY_ID_READ), EN(ERR_FRAME_CONTENT_SIZE_READ), EN(ERR_SKIP_FRAME),
    EN(ERR_WINDOW_TOO_BIG), EN(ERR_WINDOW_TOO_SMALL), EN(ERR_WINDOW_SIZE_TOO_BIG), EN(ERR_DICT_NOT_PROVIDED), EN(ERR_NOT_YET_INITIALIZED),
    EN(ERR_FAILED_TO_READ_CHECKSUM), EN(ERR_FAILED_TO_DRAIN_DECODEBUFFER), EN(ERR_FAILED_TO_SKIP_FRAME), EN(ERR_TARGET_TOO_SMALL),
    EN(ERR_BLOCK_HEADER_READ), EN(ERR_FOUND_RESERVED_BLOCK), EN(ERR_BLOCK_SIZE_TOO_LARGE), EN(ERR_DECODER_STATE_IS_FAILED),
    EN(ERR_EXPECTED_HEADER_OF_PREVIOUS_BLOCK), EN(ERR_BLOCK_BODY_READ), EN(ERR_BLOCK_CONTENT_READ), EN(ERR_MALFORMED_SECTION_HEADER),
    EN(ERR_LITSEC_ILLEGAL_TYPE), EN(ERR_LITSEC_GET_BITS), EN(ERR_LITSEC_NOT_ENOUGH_BYTES), EN(ERR_SEQHDR_NOT_ENOUGH_BYTES),
    EN(ERR_LIT_MISSING_COMPRESSED_SIZE), EN(ERR_LIT_MISSING_NUM_STREAMS), EN(ERR_LIT_GET_BITS), EN(ERR_LIT_UNINITIALIZED_HUFFMAN_TABLE),
    EN(ERR_LIT_MISSING_BYTES_FOR_JUMP_HEADER), EN(ERR_LIT_MISSING_BYTES_FOR_LITERALS), EN(ERR_LIT_EXTRA_PADDING),
    EN(ERR_LIT_BITSTREAM_READ_MISMATCH), EN(ERR_LIT_DECODED_LITERAL_COUNT_MISMATCH), EN(ERR_HUF_GET_BITS), EN(ERR_HUF_FSE_DECODER),
    EN(ERR_HUF_SOURCE_IS_EMPTY), EN(ERR_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS), EN(ERR_HUF_EXTRA_PADDING), EN(ERR_HUF_TOO_MANY_WEIGHTS),
    EN(ERR_HUF_MISSING_WEIGHTS), EN(ERR_HUF_LEFTOVER_NOT_POWER_OF_2), EN(ERR_HUF_NOT_ENOUGH_BYTES_TO_DECOMPRESS_WEIGHTS),
    EN(ERR_HUF_FSE_TABLE_USED_TOO_MANY_BYTES), EN(ERR_HUF_NOT_ENOUGH_BYTES_IN_SOURCE), EN(ERR_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS),
    EN(ERR_HUF_MAX_BITS_TOO_HIGH), EN(ERR_FSE_ACC_LOG_IS_ZERO), EN(ERR_FSE_ACC_LOG_TOO_BIG), EN(ERR_FSE_GET_BITS),
    EN(ERR_FSE_PROBABILITY_COUNTER_MISMATCH), EN(ERR_FSE_TOO_MANY_SYMBOLS), EN(ERR_FSE_TABLE_IS_UNINITIALIZED), EN(ERR_SEQ_EXTRA_PADDING),
    EN(ERR_SEQ_UNSUPPORTED_OFFSET), EN(ERR_SEQ_ZERO_OFFSET), EN(ERR_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES), EN(ERR_SEQ_EXTRA_BITS),
    EN(ERR_SEQ_MISSING_COMPRESSION_MODE), EN(ERR_SEQ_MISSING_BYTE_FOR_RLE_LL_TABLE), EN(ERR_SEQ_MISSING_BYTE_FOR_RLE_OF_TABLE),
    EN(ERR_SEQ_MISSING_BYTE_FOR_RLE_ML_TABLE), EN(ERR_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE), EN(ERR_EXEC_ZERO_OFFSET),
    EN(ERR_EXEC_NOT_ENOUGH_BYTES_IN_DICTIONARY), EN(ERR_EXEC_OFFSET_TOO_BIG), EN(ERR_DICT_NOT_ENOUGH_BYTES), EN(ERR_DICT_BAD_MAGIC_NUM),
    EN(ERR_REFERENCE_WOULD_PANIC), EN(ERR_BLOCK_OUTPUT_LIMIT), EN(ERR_INVALID_ARGUMENT), EN(ERR_OUT_OF_MEMORY), EN(ERR_NO_DEVICE), EN(ERR_CUDA),
};
#undef EN

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    // contents are NOT preserved
    int ensure(size_t n, bool grow = true) {
        if (n <= cap) return 0;
        size_t want = n;
        if (grow && cap) want = std::max(n, cap + cap / 2);
        release();
        if (cudaMalloc(&p, want ? want : 16) != cudaSuccess) { p = nullptr; cudaGetLastError(); return B200Z_ERR_OUT_OF_MEMORY; }
        cap = want ? want : 16;
        return 0;
    }
    template <class T> T *as() const { return (T *)p; }
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
struct b200z_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t side = nullptr;          // k_huf runs here, beside k_fse
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    struct PipeResources *pipe = nullptr;  // lazily created by the pipelined one-shot path
    struct CompressResources *comp = nullptr;  // lazily created by the first compression call
    FseSlot *d_predef = nullptr;
    std::string err;
    uint64_t launches = 0;
    uint32_t flags = 0;
    uint32_t match_ctas = 0;              // resident k_cmatch CTAs on this device (init_compress_kernels)
    int set_cuda_err(cudaError_t e, const char *what) {
        char buf[256];
        snprintf(buf, sizeof buf, "CUDA error in %s: %s", what, cudaGetErrorString(e));
        err = buf;
        cudaGetLastError();
        return B200Z_ERR_CUDA;
    }
    int use() { cudaError_t e = cudaSetDevice(device); return e == cudaSuccess ? 0 : set_cuda_err(e, "cudaSetDevice"); }
};

#define CU(ctx, call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return (ctx)->set_cuda_err(_e, #call); } while (0)

extern "C" const char *b200z_error_name(int code) {
    for (const auto &e : kErrNames) if (e.code == code) return e.name;
    return "UNKNOWN";
}
extern "C" int b200z_abi_version(void) { return B200Z_ABI_VERSION; }

extern "C" int b200z_ctx_create(int device, b200z_ctx **out) {
    if (!out) return B200Z_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) { cudaGetLastError(); return B200Z_ERR_NO_DEVICE; }
    std::unique_ptr<b200z_ctx> c(new b200z_ctx());
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_NO_DEVICE; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_NO_DEVICE; }
    if (cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_lo) != cudaSuccess || cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_CUDA; }
    if (cudaMalloc((void **)&c->d_predef, sizeof(FseSlot)) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_OUT_OF_MEMORY; }
    if (init_kernels() || init_compress_kernels(&c->match_ctas)) { cudaGetLastError(); return B200Z_ERR_CUDA; }
    int e = launch_predefined(c->d_predef, c->stream);
    if (e || cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_CUDA; }
    c->launches = 1;
    *out = c.release();
    return 0;
}
static void pipe_free(b200z_ctx *c);
static void comp_free(b200z_ctx *c);
extern "C" void b200z_ctx_destroy(b200z_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    pipe_free(c);
    comp_free(c);
    if (c->d_predef) cudaFree(c->d_predef);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}
extern "C" const char *b200z_ctx_last_error_message(const b200z_ctx *c) { return c ? c->err.c_str() : ""; }
extern "C" void *b200z_ctx_stream(const b200z_ctx *c) { return c ? (void *)c->stream : nullptr; }
extern "C" uint64_t b200z_ctx_kernel_launches(const b200z_ctx *c) { return c ? c->launches : 0; }
extern "C" void b200z_ctx_set_flags(b200z_ctx *c, uint32_t flags) { if (c) c->flags = flags; }
extern "C" uint32_t b200z_ctx_flags(const b200z_ctx *c) { return c ? c->flags : 0; }
extern "C" uint64_t b200z_xxh64(const uint8_t *data, size_t len) { XXH64State s; s.reset(); s.update(data, len); return s.digest(); }

// ---------------------------------------------------------------------------------------------------------------
// dictionaries
// ---------------------------------------------------------------------------------------------------------------
struct b200z_dict {
    b200z_ctx *ctx = nullptr;
    uint32_t id = 0;
    uint32_t hist[3] = {1, 4, 8};
    bool has_tables = false;
    HufSlot *d_huf = nullptr;
    FseSlot *d_fse = nullptr;
    uint8_t *d_content = nullptr;
    size_t content_len = 0;
};

static void dict_free(b200z_dict *d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    if (d->d_huf) cudaFree(d->d_huf);
    if (d->d_fse) cudaFree(d->d_fse);
    if (d->d_content) cudaFree(d->d_content);
    delete d;
}

static int dict_upload_content(b200z_dict *d, const uint8_t *content, size_t len) {
    b200z_ctx *c = d->ctx;
    d->content_len = len;
    CU(c, cudaMalloc((void **)&d->d_content, len + 16));
    if (len) CU(c, cudaMemcpy(d->d_content, content, len, cudaMemcpyHostToDevice));
    return 0;
}

// Dictionary::decode_dict (dictionary.rs:45-126).  The table descriptions are parsed and expanded with the same
// code the GPU runs per block (tables.cuh, compiled for the host here) and uploaded once.
extern "C" int b200z_dict_create(b200z_ctx *c, const uint8_t *raw, size_t len, b200z_dict **out) {
    if (!c || !out || (!raw && len)) return B200Z_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (int e = c->use()) return e;
    if (len < 8) return B200Z_ERR_DICT_NOT_ENOUGH_BYTES;
    static const uint8_t magic[4] = {0x37, 0xA4, 0x30, 0xEC};
    if (memcmp(raw, magic, 4) != 0) return B200Z_ERR_DICT_BAD_MAGIC_NUM;
    std::unique_ptr<b200z_dict, void (*)(b200z_dict *)> d(new b200z_dict(), dict_free);
    d->ctx = c;
    d->id = (uint32_t)raw[4] | ((uint32_t)raw[5] << 8) | ((uint32_t)raw[6] << 16) | ((uint32_t)raw[7] << 24);
    const uint8_t *t = raw + 8;
    size_t tl = len - 8;
    std::unique_ptr<HufSlot> huf(new HufSlot());
    std::unique_ptr<FseSlot> fse(new FseSlot());
    memset(huf.get(), 0, sizeof(HufSlot));
    memset(fse.get(), 0, sizeof(FseSlot));
    uint32_t used = 0;
    int e = huf_build_decoder(t, (uint32_t)std::min<size_t>(tl, 0x7fffffff), huf.get(), used);
    if (e) return e;
    if (tl < used) return B200Z_ERR_DICT_NOT_ENOUGH_BYTES;
    t += used; tl -= used;
    struct { FseTab *tab; uint32_t max_log, max_sym; } order[3] = {{&fse->of, 8, 31}, {&fse->ml, 9, 52}, {&fse->ll, 9, 35}};  // OF, ML, LL
    for (auto &o : order) {
        e = fse_build_decoder(t, (uint32_t)std::min<size_t>(tl, 0x7fffffff), o.max_log, o.max_sym, o.tab, used);
        if (e) return e;
        if (tl < used) return B200Z_ERR_DICT_NOT_ENOUGH_BYTES;
        t += used; tl -= used;
    }
    if (tl < 12) return B200Z_ERR_DICT_NOT_ENOUGH_BYTES;
    for (int i = 0; i < 3; i++) d->hist[i] = (uint32_t)t[4 * i] | ((uint32_t)t[4 * i + 1] << 8) | ((uint32_t)t[4 * i + 2] << 16) | ((uint32_t)t[4 * i + 3] << 24);
    d->has_tables = true;
    CU(c, cudaMalloc((void **)&d->d_huf, sizeof(HufSlot)));
    CU(c, cudaMalloc((void **)&d->d_fse, sizeof(FseSlot)));
    CU(c, cudaMemcpy(d->d_huf, huf.get(), sizeof(HufSlot), cudaMemcpyHostToDevice));
    CU(c, cudaMemcpy(d->d_fse, fse.get(), sizeof(FseSlot), cudaMemcpyHostToDevice));
    if ((e = dict_upload_content(d.get(), t + 12, tl - 12))) return e;
    *out = d.release();
    return 0;
}
extern "C" int b200z_dict_create_raw_content(b200z_ctx *c, uint32_t id, const uint8_t *content, size_t len, b200z_dict **out) {
    if (!c || !out || (!content && len)) return B200Z_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (int e = c->use()) return e;
    std::unique_ptr<b200z_dict, void (*)(b200z_dict *)> d(new b200z_dict(), dict_free);
    d->ctx = c; d->id = id;
    if (int e = dict_upload_content(d.get(), content, len)) return e;
    *out = d.release();
    return 0;
}
extern "C" uint32_t b200z_dict_id(const b200z_dict *d) { return d ? d->id : 0; }
extern "C" int b200z_dict_offset_history(const b200z_dict *d, uint32_t out[3]) { if (!d) return B200Z_ERR_INVALID_ARGUMENT; memcpy(out, d->hist, 12); return 0; }
extern "C" size_t b200z_dict_content_size(const b200z_dict *d) { return d ? d->content_len : 0; }
extern "C" void b200z_dict_destroy(b200z_dict *d) { dict_free(d); }

// ---------------------------------------------------------------------------------------------------------------
// A "submission": host-side plan + its device mirror.  Used by the batch entry (many frames, fresh state) and
// by the FrameDecoder mirror (one frame, a few new blocks, state carried on the device).
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct CarrySet { const HufSlot *huf = nullptr; const FseTab *ll = nullptr, *of = nullptr, *ml = nullptr; };

struct Submission {
    std::vector<BlockDesc> descs;
    std::vector<BlockRefs> refs;
    std::vector<FrameDesc> frames;
    std::vector<FrameState> states;
    std::vector<CarrySet> carries;   // TabRef::CARRY idx -> device tables (dictionaries / streaming carry)
    uint32_t n_huf = 0, n_fse = 0;
    uint64_t lit_bytes = 0, nseq = 0;
    DevBuf d_descs, d_aux, d_frames, d_states, d_huf, d_fse, d_lit, d_seq, d_sched, d_order;
    std::vector<uint32_t> fse_order;    // PipelineArgs::fse_order (empty: descriptor order)
    std::vector<uint32_t> cta_frames;   // frames executed by k_exec_cta (the rest: k_exec, one warp per frame)
    std::vector<uint32_t> sched_image;  // host copy of the initial ticket / resume[] image (kept alive for the async upload)

    void clear() {
        descs.clear(); refs.clear(); frames.clear(); states.clear(); carries.clear();
        n_huf = n_fse = 0; lit_bytes = 0; nseq = 0;
    }
    // resolve table references to device pointers and upload descriptors
    int upload(b200z_ctx *c, cudaStream_t stream = nullptr) {
        if (!stream) stream = c->stream;
        int e;
        if ((e = d_descs.ensure(descs.size() * sizeof(BlockDesc)))) return e;
        if ((e = d_aux.ensure(descs.size() * sizeof(BlockAux)))) return e;
        if ((e = d_frames.ensure(frames.size() * sizeof(FrameDesc)))) return e;
        if ((e = d_states.ensure(states.size() * sizeof(FrameState)))) return e;
        if ((e = d_huf.ensure((size_t)n_huf * sizeof(HufSlot)))) return e;
        if ((e = d_fse.ensure((size_t)n_fse * sizeof(FseSlot)))) return e;
        if ((e = d_lit.ensure(lit_bytes + 64))) return e;
        if ((e = d_seq.ensure((nseq + 4) * 12))) return e;
        // which execution kernel takes a frame (route_exec_frames, plan.cpp): single-block frames, tiny frames and frames with a
        // dictionary always stay with the warp kernel (dictionary reach is its exact path); the multi-block frames go to k_exec_cta
        // or k_exec by a cost model on sequences + compressed bytes.  B200Z_EXEC_MODE = warp | cta | auto (default) overrides for
        // tests and measurements.
        cta_frames.clear();
        {
            const char *m = getenv("B200Z_EXEC_MODE");
            const bool force_warp = m && !strcmp(m, "warp"), force_cta = m && !strcmp(m, "cta");
            std::vector<uint64_t> work(frames.size(), 0);
            std::vector<uint8_t> eligible(frames.size(), 0);
            for (size_t f = 0; f < frames.size() && !force_warp; f++) {
                const FrameDesc &fd = frames[f];
                if (fd.nblocks == 0) continue;
                uint64_t src = 0, nseq = 0;
                for (uint32_t k = 0; k < fd.nblocks; k++) { src += descs[fd.first_block + k].src_size; nseq += descs[fd.first_block + k].nseq; }
                work[f] = nseq + src / 16;
                if (fd.dict) continue;
                if (force_cta) cta_frames.push_back((uint32_t)f);
                else eligible[f] = fd.nblocks >= 2 && src >= 4096;
            }
            if (!force_warp && !force_cta) route_exec_frames(work.data(), eligible.data(), frames.size(), num_sms(), cta_frames);
        }
        // the order in which k_fse takes the blocks (build_fse_order, plan.cpp).  B200Z_FSE_ORDER=0 keeps the descriptor order.
        fse_order.clear();
        {
            const char *eo = getenv("B200Z_FSE_ORDER");
            if (!(eo && eo[0] == '0') && !frames.empty()) {
                std::vector<uint8_t> on_cta(frames.size(), 0);
                for (uint32_t f : cta_frames) on_cta[f] = 1;
                std::vector<uint32_t> fb(frames.size()), nb(frames.size()), nseq(descs.size());
                for (size_t f = 0; f < frames.size(); f++) { fb[f] = frames[f].first_block; nb[f] = frames[f].nblocks; }
                for (size_t i = 0; i < descs.size(); i++) nseq[i] = descs[i].nseq;
                build_fse_order(fb.data(), nb.data(), on_cta.data(), frames.size(), nseq.data(), descs.size(), fse_order);
            }
            if (!fse_order.empty() && (e = d_order.ensure(4 * fse_order.size()))) return e;
        }
        // scheduling buffer: [ticket + 3 counters][resume[nframes]][cta frame list][initial image of the first two parts]
        if ((e = d_sched.ensure(2 * (16 + 4 * frames.size()) + 4 * cta_frames.size() + 32))) return e;
        HufSlot *hs = d_huf.as<HufSlot>();
        FseSlot *fs = d_fse.as<FseSlot>();
        const FseSlot *pd = c->d_predef;
        for (size_t i = 0; i < descs.size(); i++) {
            BlockDesc &d = descs[i];
            const BlockRefs &r = refs[i];
            auto huf = [&](const TabRef &t) -> const HufSlot * {
                if (t.kind == TabRef::SLOT) return hs + t.idx;
                if (t.kind == TabRef::CARRY) return carries[t.idx].huf;
                return nullptr;
            };
            auto fse = [&](const TabRef &t, int which) -> const FseTab * {
                if (t.kind == TabRef::SLOT) return which == 0 ? &fs[t.idx].ll : (which == 1 ? &fs[t.idx].of : &fs[t.idx].ml);
                if (t.kind == TabRef::PREDEF) return which == 0 ? &pd->ll : (which == 1 ? &pd->of : &pd->ml);
                if (t.kind == TabRef::CARRY) return which == 0 ? carries[t.idx].ll : (which == 1 ? carries[t.idx].of : carries[t.idx].ml);
                return nullptr;
            };
            d.huf = huf(r.huf);
            d.huf_build = r.build_huf >= 0 ? hs + r.build_huf : nullptr;
            d.ll = fse(r.ll, 0); d.of = fse(r.of, 1); d.ml = fse(r.ml, 2);
            d.fse_build = r.build_fse >= 0 ? fs + r.build_fse : nullptr;
        }
        if (!descs.empty()) CU(c, cudaMemcpyAsync(d_descs.p, descs.data(), descs.size() * sizeof(BlockDesc), cudaMemcpyHostToDevice, stream));
        if (!frames.empty()) CU(c, cudaMemcpyAsync(d_frames.p, frames.data(), frames.size() * sizeof(FrameDesc), cudaMemcpyHostToDevice, stream));
        if (!states.empty()) CU(c, cudaMemcpyAsync(d_states.p, states.data(), states.size() * sizeof(FrameState), cudaMemcpyHostToDevice, stream));
        if (!fse_order.empty()) CU(c, cudaMemcpyAsync(d_order.p, fse_order.data(), 4 * fse_order.size(), cudaMemcpyHostToDevice, stream));
        if (!cta_frames.empty())
            CU(c, cudaMemcpyAsync(d_sched.as<uint8_t>() + 16 + 4 * frames.size(), cta_frames.data(), 4 * cta_frames.size(), cudaMemcpyHostToDevice, stream));
        if (!frames.empty()) {
            sched_image.assign(4 + frames.size(), 0u);
            for (uint32_t f : cta_frames) sched_image[4 + f] = RESUME_SKIP;   // not for the first k_exec launch; k_exec_cta rewrites it
            CU(c, cudaMemcpyAsync(d_sched.as<uint8_t>() + 16 + 4 * (frames.size() + cta_frames.size()), sched_image.data(), 4 * sched_image.size(), cudaMemcpyHostToDevice, stream));
        }
        return 0;
    }
    PipelineArgs args(const uint8_t *d_input, uint8_t *d_output, uint64_t out_cap) const {
        PipelineArgs a;
        a.descs = d_descs.as<BlockDesc>(); a.aux = d_aux.as<BlockAux>(); a.frames = d_frames.as<FrameDesc>(); a.states = d_states.as<FrameState>();
        a.input = d_input; a.lit_scratch = d_lit.as<uint8_t>(); a.seq_scratch = d_seq.as<uint32_t>();
        a.output = d_output; a.output_cap = out_cap; a.nblocks = (uint32_t)descs.size(); a.nframes = (uint32_t)frames.size();
        uint8_t *sp = d_sched.as<uint8_t>();
        a.ticket = (uint32_t *)sp; a.resume = (uint32_t *)(sp + 16); a.cta_frames = (const uint32_t *)(sp + 16 + 4 * frames.size());
        a.n_cta_frames = (uint32_t)cta_frames.size(); a.sched_bytes = (uint32_t)(16 + 4 * frames.size());
        a.sched_init = (const uint32_t *)(sp + 16 + 4 * (frames.size() + cta_frames.size()));
        a.fse_order = fse_order.empty() ? nullptr : d_order.as<uint32_t>();
        return a;
    }
};

// initial cursor of a frame: fresh, or the dictionary's tables (scratch.rs:70-78)
void cursor_from_carry(TableCursor &cur, const CarrySet &cs, uint32_t carry_idx) {
    cur = TableCursor();
    if (cs.huf) { cur.huf.kind = TabRef::CARRY; cur.huf.idx = carry_idx; }
    if (cs.ll) { cur.ll.kind = TabRef::CARRY; cur.ll.idx = carry_idx; }
    if (cs.of) { cur.of.kind = TabRef::CARRY; cur.of.idx = carry_idx; }
    if (cs.ml) { cur.ml.kind = TabRef::CARRY; cur.ml.idx = carry_idx; }
}
CarrySet carry_of_dict(const b200z_dict *d) {
    CarrySet cs;
    if (d && d->has_tables) { cs.huf = d->d_huf; cs.ll = &d->d_fse->ll; cs.of = &d->d_fse->of; cs.ml = &d->d_fse->ml; }
    return cs;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// tier 1: batch
// ---------------------------------------------------------------------------------------------------------------
struct FramePlanInfo {
    int pre_status = 0, pre_stage = 0;       // failure before any block (frame header / window / dictionary)
    FrameHeader hdr;
    uint64_t window = 0;
    uint64_t bytes_read_full = 0;            // bytes_read_from_source after a fully successful decode
    size_t first_block_end = 0;              // index into block_end_bytes
    bool has_checksum = false;
    uint32_t checksum = 0;
    uint32_t skip_len = 0;
    int32_t sub_frame = -1;                  // index in Submission::frames, -1 if the frame never reaches the GPU
};

struct b200z_batch {
    b200z_ctx *ctx = nullptr;
    Submission sub;
    std::vector<FramePlanInfo> info;
    std::vector<uint64_t> block_end_bytes;   // per planned block: bytes_read_from_source after that block
    DevBuf d_input_own;
    const uint8_t *d_input = nullptr;
    DevBuf d_states_init;
    size_t input_len = 0;
    bool ran = false;
    bool checksummed = false;
};

// what k_walk brought back for a batch whose input lives in device memory (the planner then never sees the compressed bytes)
struct WalkHost { std::vector<WalkFrame> wf; std::vector<WalkBlock> wb; std::vector<uint32_t> first; };

static int plan_batch(b200z_batch *b, const uint8_t *in, size_t in_len, const b200z_frame_io *frames, size_t nframes,
                      const b200z_dict *const *dicts, size_t ndicts, const b200z_dict *forced, uint64_t max_window, const WalkHost *walk = nullptr) {
    Submission &s = b->sub;
    s.clear();
    b->info.assign(nframes, FramePlanInfo());
    b->block_end_bytes.clear();
    if (max_window == 0) max_window = B200Z_DEFAULT_MAX_WINDOW_SIZE;
    max_window = std::min<uint64_t>(max_window, (1ull << 41) + 7 * (1ull << 38));
    // carry sets: one per dictionary (+ forced)
    std::vector<const b200z_dict *> dlist(dicts, dicts + ndicts);
    int forced_idx = -1;
    if (forced) {
        auto it = std::find(dlist.begin(), dlist.end(), forced);
        if (it == dlist.end()) { dlist.push_back(forced); forced_idx = (int)dlist.size() - 1; } else forced_idx = (int)(it - dlist.begin());
    }
    for (auto *d : dlist) s.carries.push_back(carry_of_dict(d));

    for (size_t i = 0; i < nframes; i++) {
        FramePlanInfo &fi = b->info[i];
        const b200z_frame_io &io = frames[i];
        if (io.src_off > in_len || io.src_size > in_len - io.src_off) { fi.pre_status = B200Z_ERR_INVALID_ARGUMENT; continue; }
        // host input: the frame's bytes; device input: the bytes the header walk picked (frame header here, block digests below)
        const uint8_t *p = walk ? walk->wf[i].hdr : in + io.src_off;
        size_t len = io.src_size, consumed = 0;
        uint32_t wk = walk ? walk->first[i] : 0;   // next block digest of this frame
        const uint32_t wk_end = walk ? wk + walk->wf[i].nblocks : 0;
        int e = parse_frame_header(p, len, fi.hdr, fi.skip_len, consumed);
        if (e) { fi.pre_status = e; fi.pre_stage = B200Z_STAGE_FRAME_HEADER; fi.bytes_read_full = consumed; continue; }
        if ((e = frame_window_size(fi.hdr, fi.window))) { fi.pre_status = e; fi.pre_stage = B200Z_STAGE_FRAME_HEADER; continue; }
        if (fi.window > max_window) { fi.pre_status = B200Z_ERR_WINDOW_SIZE_TOO_BIG; fi.pre_stage = B200Z_STAGE_FRAME_HEADER; continue; }
        int dict_idx = -1;
        if (fi.hdr.has_dict_id) {
            for (size_t k = 0; k < dlist.size() && k < ndicts; k++) if (dlist[k]->id == fi.hdr.dict_id) dict_idx = (int)k;
            if (dict_idx < 0) { fi.pre_status = B200Z_ERR_DICT_NOT_PROVIDED; fi.pre_stage = B200Z_STAGE_FRAME_HEADER; continue; }
        }
        if (forced_idx >= 0) dict_idx = forced_idx;
        const b200z_dict *dict = dict_idx >= 0 ? dlist[dict_idx] : nullptr;

        FrameDesc fd;
        memset(&fd, 0, sizeof fd);
        fd.out_off = io.out_off; fd.out_cap = io.out_cap; fd.window_size = fi.window;
        fd.dict = dict ? dict->d_content : nullptr; fd.dict_len = dict ? dict->content_len : 0;
        fd.first_block = (uint32_t)s.descs.size();
        FrameState st;
        memset(&st, 0, sizeof st);
        st.hist[0] = dict ? dict->hist[0] : 1; st.hist[1] = dict ? dict->hist[1] : 4; st.hist[2] = dict ? dict->hist[2] : 8;
        TableCursor cur;
        if (dict_idx >= 0) cursor_from_carry(cur, s.carries[dict_idx], (uint32_t)dict_idx);
        fi.first_block_end = b->block_end_bytes.size();

        uint64_t pos = consumed, bytes_read = consumed;
        uint32_t bif = 0;
        for (;;) {
            if (len - pos < 3) { fd.host_status = mk_status(B200Z_ERR_BLOCK_HEADER_READ, B200Z_STAGE_BLOCK_HEADER); break; }
            BlockHeader bh;
            const WalkBlock *wbk = nullptr;
            if (walk) {
                if (wk >= wk_end || walk->wb[wk].pos != pos) return B200Z_ERR_INVALID_ARGUMENT;   // (the walk and the planner follow the same chain)
                wbk = &walk->wb[wk++];
            }
            if ((e = parse_block_header(wbk ? wbk->bh : p + pos, bh))) { fd.host_status = mk_status((uint32_t)e, B200Z_STAGE_BLOCK_HEADER); break; }
            pos += 3;
            if (len - pos < bh.content_size) {
                fd.host_status = mk_status(bh.type == BT_COMPRESSED ? B200Z_ERR_BLOCK_CONTENT_READ : B200Z_ERR_BLOCK_BODY_READ, B200Z_STAGE_BLOCK_BODY);
                break;
            }
            BlockDesc d;
            memset(&d, 0, sizeof d);
            BlockRefs r;
            d.src_off = io.src_off + pos; d.src_size = bh.content_size; d.frame = (uint32_t)s.frames.size();
            d.btype = bh.type; d.raw_size = bh.decompressed_size; d.block_in_frame = bif++; d.last = bh.last;
            if (bh.type == BT_COMPRESSED) {
                if (wbk) plan_compressed_block_view(wbk->lit, wbk->seq, bh.content_size, d, r, cur, s.n_huf, s.n_fse, s.lit_bytes, s.nseq);
                else plan_compressed_block(p + pos, bh.content_size, d, r, cur, s.n_huf, s.n_fse, s.lit_bytes, s.nseq);
            }
            pos += bh.content_size;
            bytes_read += 3 + bh.content_size;
            s.descs.push_back(d); s.refs.push_back(r);
            b->block_end_bytes.push_back(bytes_read);
            if (d.host_status) break;  // the reference stops here; later blocks are never looked at
            if (bh.last) {
                if (fi.hdr.content_checksum()) {
                    if (len - pos < 4) { fd.host_status = mk_status(B200Z_ERR_FAILED_TO_READ_CHECKSUM, B200Z_STAGE_CHECKSUM); break; }
                    fi.has_checksum = true;
                    if (walk && (walk->wf[i].end_pos != pos || walk->wf[i].tail_avail < 4)) return B200Z_ERR_INVALID_ARGUMENT;
                    const uint8_t *q = walk ? walk->wf[i].tail : p + pos;
                    fi.checksum = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
                    bytes_read += 4;
                }
                break;
            }
        }
        fd.nblocks = (uint32_t)s.descs.size() - fd.first_block;
        fi.bytes_read_full = bytes_read;
        fi.sub_frame = (int32_t)s.frames.size();
        s.frames.push_back(fd); s.states.push_back(st);
    }
    return 0;
}

// k_walk twice (count, fill) with a host prefix sum in between; ~16 bytes per block and 48 per frame come back
static int device_walk(b200z_ctx *c, const uint8_t *d_input, size_t input_len, const b200z_frame_io *frames, size_t nframes, WalkHost &w) {
    w.wf.assign(nframes, WalkFrame()); w.first.assign(nframes, 0); w.wb.clear();
    if (!nframes) return 0;
    std::vector<uint64_t> so(2 * nframes);
    for (size_t i = 0; i < nframes; i++) { so[i] = frames[i].src_off; so[nframes + i] = frames[i].src_size; }
    DevBuf d_io, d_wf, d_first, d_wb;
    if (int e = d_io.ensure(so.size() * 8, false)) return e;
    if (int e = d_wf.ensure(nframes * sizeof(WalkFrame), false)) return e;
    if (int e = d_first.ensure(nframes * 4, false)) return e;
    CU(c, cudaMemcpyAsync(d_io.p, so.data(), so.size() * 8, cudaMemcpyHostToDevice, c->stream));
    const uint64_t *d_off = d_io.as<uint64_t>(), *d_sz = d_off + nframes;
    int le = launch_walk(d_input, input_len, d_off, d_sz, (uint32_t)nframes, d_wf.as<WalkFrame>(), nullptr, nullptr, 0, c->stream);
    if (le) return c->set_cuda_err((cudaError_t)le, "k_walk");
    CU(c, cudaMemcpyAsync(w.wf.data(), d_wf.p, nframes * sizeof(WalkFrame), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    uint64_t total = 0;
    for (size_t i = 0; i < nframes; i++) { w.first[i] = (uint32_t)total; total += w.wf[i].nblocks; }
    if (total > 0xFFFFFFF0ull) return B200Z_ERR_INVALID_ARGUMENT;
    c->launches += 1;
    if (!total) return 0;
    w.wb.resize(total);
    if (int e = d_wb.ensure(total * sizeof(WalkBlock), false)) return e;
    CU(c, cudaMemcpyAsync(d_first.p, w.first.data(), nframes * 4, cudaMemcpyHostToDevice, c->stream));
    le = launch_walk(d_input, input_len, d_off, d_sz, (uint32_t)nframes, d_wf.as<WalkFrame>(), d_first.as<uint32_t>(), d_wb.as<WalkBlock>(), 1, c->stream);
    if (le) return c->set_cuda_err((cudaError_t)le, "k_walk");
    CU(c, cudaMemcpyAsync(w.wb.data(), d_wb.p, total * sizeof(WalkBlock), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    c->launches += 1;
    return 0;
}

extern "C" int b200z_batch_prepare(b200z_ctx *c, const uint8_t *input, size_t input_len, int input_mem, const b200z_frame_io *frames,
                                   size_t nframes, const b200z_dict *const *dicts, size_t ndicts, const b200z_dict *forced,
                                   uint64_t max_window, b200z_batch **out) {
    if (!c || !out || (!input && input_len) || (!frames && nframes) || (!dicts && ndicts)) return B200Z_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (int e = c->use()) return e;
    std::unique_ptr<b200z_batch> b(new b200z_batch());
    b->ctx = c; b->input_len = input_len;
    const uint8_t *hin = input;
    WalkHost walk;
    std::vector<uint8_t> host_copy;
    if (input_mem == B200Z_MEM_DEVICE) {
        // The input stays on the device: k_walk follows the frame / block / section headers there and brings back the ~16 bytes per
        // block the planner parses (SURVEY.md 8(f).3) -- not the compressed data (B200Z_WALK=host copies it back and walks on the host,
        // for A/B tests).
        b->d_input = input;
        const char *wm = getenv("B200Z_WALK");
        if (wm && !strcmp(wm, "host")) {
            host_copy.resize(input_len);
            if (input_len) CU(c, cudaMemcpy(host_copy.data(), input, input_len, cudaMemcpyDeviceToHost));
            hin = host_copy.data();
        } else {
            hin = nullptr;
            if (int e = device_walk(c, input, input_len, frames, nframes, walk)) return e;
        }
    }
    if (int e = plan_batch(b.get(), hin, input_len, frames, nframes, dicts, ndicts, forced, max_window, hin ? nullptr : (input_mem == B200Z_MEM_DEVICE ? &walk : nullptr))) return e;
    if (input_mem != B200Z_MEM_DEVICE) {
        if (int e = b->d_input_own.ensure(input_len + 16, false)) return e;
        if (input_len) CU(c, cudaMemcpyAsync(b->d_input_own.p, input, input_len, cudaMemcpyHostToDevice, c->stream));
        b->d_input = b->d_input_own.as<uint8_t>();
    }
    if (int e = b->sub.upload(c)) return e;
    if (int e = b->d_states_init.ensure(b->sub.states.size() * sizeof(FrameState), false)) return e;
    if (!b->sub.states.empty())
        CU(c, cudaMemcpyAsync(b->d_states_init.p, b->sub.states.data(), b->sub.states.size() * sizeof(FrameState), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    *out = b.release();
    return 0;
}

extern "C" int b200z_batch_run(b200z_batch *b, uint8_t *d_output, size_t output_cap) {
    if (!b) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    if (int e = c->use()) return e;
    Submission &s = b->sub;
    if (!s.states.empty())
        CU(c, cudaMemcpyAsync(s.d_states.p, b->d_states_init.p, s.states.size() * sizeof(FrameState), cudaMemcpyDeviceToDevice, c->stream));
    PipelineArgs a = s.args(b->d_input, d_output, output_cap);
    PipelineStreams ps{c->stream, c->side, c->ev_fork, c->ev_join};
    int e = launch_pipeline_overlapped(a, ps);
    if (e) return c->set_cuda_err((cudaError_t)e, "launch_pipeline");
    c->launches += pipeline_launch_count(a);
    b->checksummed = false;
    if ((c->flags & B200Z_FLAG_CHECKSUM) && a.nframes) {
        if ((e = launch_checksum(a, c->stream))) return c->set_cuda_err((cudaError_t)e, "launch_checksum");
        c->launches += 1;
        b->checksummed = true;
    }
    b->ran = true;
    return 0;
}

// Same as b200z_batch_run but with a CUDA event between stages; synchronises and reports per-kernel milliseconds.
extern "C" int b200z_batch_run_profile(b200z_batch *b, uint8_t *d_output, size_t output_cap, float *stage_ms, size_t nstages) {
    if (!b || !stage_ms) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    if (int e = c->use()) return e;
    Submission &s = b->sub;
    if (!s.states.empty())
        CU(c, cudaMemcpyAsync(s.d_states.p, b->d_states_init.p, s.states.size() * sizeof(FrameState), cudaMemcpyDeviceToDevice, c->stream));
    PipelineArgs a = s.args(b->d_input, d_output, output_cap);
    cudaEvent_t ev[kNumStages + 1];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    if (int e = reset_sched(a, c->stream)) return c->set_cuda_err((cudaError_t)e, "reset_sched");
    CU(c, cudaEventRecord(ev[0], c->stream));
    for (int st = 0; st < kNumStages; st++) {
        int e = launch_stage(a, st, c->stream);
        if (e) return c->set_cuda_err((cudaError_t)e, "launch_stage");
        CU(c, cudaEventRecord(ev[st + 1], c->stream));
    }
    c->launches += pipeline_launch_count(a);
    CU(c, cudaStreamSynchronize(c->stream));
    for (int st = 0; st < kNumStages && (size_t)st < nstages; st++) CU(c, cudaEventElapsedTime(&stage_ms[st], ev[st], ev[st + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    b->ran = true;
    return 0;
}
// One pass as b200z_batch_run launches it, with events on the stream: out_ms[0] = 0, out_ms[1..3] = completion time, relative to
// the start of the pass, of the table builds + k_huf (two streams), of the pair k_fse + k_exec (k_exec runs beside k_fse as its programmatic dependent: an event
// between the two would serialise them) and of k_exec_cta + the k_exec launch that takes what it handed back.
extern "C" int b200z_batch_run_timeline(b200z_batch *b, uint8_t *d_output, size_t output_cap, float *out_ms, size_t n) {
    if (!b || !out_ms || n < 4) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    if (int e = c->use()) return e;
    Submission &s = b->sub;
    if (!s.states.empty())
        CU(c, cudaMemcpyAsync(s.d_states.p, b->d_states_init.p, s.states.size() * sizeof(FrameState), cudaMemcpyDeviceToDevice, c->stream));
    PipelineArgs a = s.args(b->d_input, d_output, output_cap);
    if (int e = reset_sched(a, c->stream)) return c->set_cuda_err((cudaError_t)e, "reset_sched");
    cudaEvent_t ev[5];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaEventRecord(ev[0], c->stream));
    PipelineStreams ps{c->stream, c->side, c->ev_fork, c->ev_join};
    CU(c, cudaEventRecord(ev[1], c->stream));
    int le = launch_tables_literals(a, ps);
    CU(c, cudaEventRecord(ev[2], c->stream));
    if (!le) le = launch_fse_exec(a, c->stream);
    CU(c, cudaEventRecord(ev[3], c->stream));
    if (!le) le = launch_cta_rest(a, c->stream);
    CU(c, cudaEventRecord(ev[4], c->stream));
    if (le) return c->set_cuda_err((cudaError_t)le, "launch_stage");
    c->launches += pipeline_launch_count(a);
    CU(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 4; i++) CU(c, cudaEventElapsedTime(&out_ms[i], ev[0], ev[i + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    return 0;
}
// host-only views of the scheduling decisions (plan.cpp), for CPU tests: no context, no device
extern "C" int b200z_debug_route_frames(const uint64_t *work, const uint8_t *eligible, size_t nframes, uint32_t sms, uint32_t *cta_frames, size_t *n_cta) {
    if ((!work || !eligible) && nframes) return B200Z_ERR_INVALID_ARGUMENT;
    if (!n_cta) return B200Z_ERR_INVALID_ARGUMENT;
    std::vector<uint32_t> out;
    route_exec_frames(work, eligible, nframes, sms, out);
    if (cta_frames) for (size_t i = 0; i < out.size(); i++) cta_frames[i] = out[i];   // room for nframes entries
    *n_cta = out.size();
    return 0;
}
extern "C" int b200z_debug_fse_order(const uint32_t *first_block, const uint32_t *nblocks, const uint8_t *on_cta, size_t nframes, const uint32_t *nseq,
                                     size_t nblocks_total, uint32_t *order, size_t *n_order) {
    if (!n_order || ((!first_block || !nblocks || !on_cta) && nframes) || (!nseq && nblocks_total)) return B200Z_ERR_INVALID_ARGUMENT;
    std::vector<uint32_t> out;
    build_fse_order(first_block, nblocks, on_cta, nframes, nseq, nblocks_total, out);
    if (order) for (size_t i = 0; i < out.size(); i++) order[i] = out[i];   // room for nblocks_total entries
    *n_order = out.size();
    return 0;
}
extern "C" int b200z_num_stages(void) { return kNumStages; }
extern "C" const char *b200z_stage_kernel_name(int stage) { return stage >= 0 && stage < kNumStages ? kStageNames[stage] : ""; }

static void fill_result(const b200z_batch *b, size_t i, const FrameState *st, b200z_frame_result &r) {
    const FramePlanInfo &fi = b->info[i];
    memset(&r, 0, sizeof r);
    r.content_size = fi.hdr.frame_content_size; r.window_size = fi.window;
    r.has_dict_id = fi.hdr.has_dict_id; r.dict_id = fi.hdr.dict_id;
    if (fi.pre_status) {
        r.status = fi.pre_status; r.stage = fi.pre_stage; r.bytes_read = fi.bytes_read_full;
        if (fi.pre_status == B200Z_ERR_SKIP_FRAME) r.content_size = fi.skip_len;
        return;
    }
    r.out_size = st->produced; r.blocks_decoded = st->blocks_done;
    if (st->status == 0) {
        r.bytes_read = fi.bytes_read_full; r.has_checksum = fi.has_checksum; r.checksum_from_data = fi.checksum;
        if (b->checksummed) { r.has_calculated_checksum = 1; r.calculated_checksum = (uint32_t)st->xxh64; }
        return;
    }
    r.status = (int32_t)(st->status & 0xffffu); r.stage = (int32_t)((st->status >> 16) & 0xffu); r.error_block = st->error_block;
    // bytes_read_from_source at the point the reference returns the error (frame_decoder.rs:325-341)
    uint32_t j = st->blocks_done;
    uint64_t before = j > 0 ? b->block_end_bytes[fi.first_block_end + j - 1] : fi.hdr.header_size;
    if (r.stage == B200Z_STAGE_BLOCK_HEADER) r.bytes_read = before;
    else if (r.stage == B200Z_STAGE_CHECKSUM) r.bytes_read = before;
    else r.bytes_read = before + 3;
}

extern "C" int b200z_batch_finish(b200z_batch *b, b200z_frame_result *results) {
    if (!b || !results) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    if (int e = c->use()) return e;
    Submission &s = b->sub;
    std::vector<FrameState> st(s.states.size());
    if (!st.empty()) CU(c, cudaMemcpyAsync(st.data(), s.d_states.p, st.size() * sizeof(FrameState), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < b->info.size(); i++) {
        int32_t sf = b->info[i].sub_frame;
        fill_result(b, i, sf >= 0 ? &st[sf] : nullptr, results[i]);
    }
    return 0;
}

extern "C" int b200z_batch_info(const b200z_batch *b, uint64_t out[8]) {
    if (!b || !out) return B200Z_ERR_INVALID_ARGUMENT;
    const Submission &s = b->sub;
    uint64_t ncomp = 0, planned = 0;
    for (auto &d : s.descs) { ncomp += d.btype == BT_COMPRESSED; planned += d.src_size + 3; }
    out[0] = s.frames.size(); out[1] = s.descs.size(); out[2] = ncomp; out[3] = planned; out[4] = s.lit_bytes; out[5] = s.nseq;
    out[6] = pipeline_launch_count(s.args(nullptr, nullptr, 0)); out[7] = 0;
    return 0;
}

extern "C" int b200z_batch_debug_literals(b200z_batch *b, uint32_t block, uint8_t *host_out, size_t cap, size_t *len) {
    if (!b || block >= b->sub.descs.size() || !len) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    const BlockDesc &d = b->sub.descs[block];
    *len = 0;
    if (d.btype != BT_COMPRESSED || (d.lit_type != LT_COMPRESSED && d.lit_type != LT_TREELESS)) return 0;
    if (cap < d.regen_size) return B200Z_ERR_TARGET_TOO_SMALL;
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(host_out, b->sub.d_lit.as<uint8_t>() + d.lit_buf_off, d.regen_size, cudaMemcpyDeviceToHost));
    *len = d.regen_size;
    return 0;
}
extern "C" int b200z_batch_debug_sequences(b200z_batch *b, uint32_t block, uint32_t *host_out, size_t cap_seqs, size_t *nseq) {
    if (!b || block >= b->sub.descs.size() || !nseq) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    const BlockDesc &d = b->sub.descs[block];
    *nseq = 0;
    if (d.btype != BT_COMPRESSED || d.nseq == 0) return 0;
    if (cap_seqs < d.nseq) return B200Z_ERR_TARGET_TOO_SMALL;
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(host_out, b->sub.d_seq.as<uint32_t>() + d.seq_buf_off * 3, (size_t)d.nseq * 12, cudaMemcpyDeviceToHost));
    // the device holds prefix sums {out_end, lit_end, of}: hand out {ll, ml, of} (of: see b200z_batch_debug_block_flags)
    uint32_t p_out = 0, p_lit = 0;
    for (size_t i = 0; i < d.nseq; i++) {
        uint32_t *r = host_out + 3 * i;
        const uint32_t oe = r[0], le = r[1], ll = le - p_lit, ml = oe - p_out - ll;
        r[0] = ll; r[1] = ml; p_out = oe; p_lit = le;
    }
    *nseq = d.nseq;
    return 0;
}
// flags of a block's sequence stage: bit 0 = `of` values are raw offset_values (otherwise offsets after do_offset_history,
// symbolic where they depend on the history at the block's start: tag << 30 | decrements, tag 1..3 = history slot + 1)
extern "C" int b200z_batch_debug_block_flags(b200z_batch *b, uint32_t block, uint32_t *flags) {
    if (!b || block >= b->sub.descs.size() || !flags) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    CU(c, cudaStreamSynchronize(c->stream));
    BlockAux ax;
    CU(c, cudaMemcpy(&ax, b->sub.d_aux.as<BlockAux>() + block, sizeof ax, cudaMemcpyDeviceToHost));
    *flags = ax.flags;
    return 0;
}
// execution scheduling counters of the LAST run: [0] frames given to k_exec_cta, [1] frames it handed back to k_exec,
// [2] OR of the reasons (1 error status, 2 capacity, 4 raw/wide sequence records, 8 block size, 16 RLE literals that do not
// fit, 32 sequence validation (dictionary reach, invalid offsets), 64 internal wait timed out, 128 frame state), [3] blocks left to k_exec
extern "C" int b200z_batch_debug_sched(b200z_batch *b, uint32_t out[4]) {
    if (!b || !out) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_ctx *c = b->ctx;
    out[0] = (uint32_t)b->sub.cta_frames.size(); out[1] = out[2] = out[3] = 0;
    if (!b->sub.d_sched.p) return 0;
    CU(c, cudaStreamSynchronize(c->stream));
    uint32_t h[4];
    CU(c, cudaMemcpy(h, b->sub.d_sched.p, sizeof h, cudaMemcpyDeviceToHost));
    out[1] = h[1]; out[2] = h[2]; out[3] = h[3];
    return 0;
}
extern "C" void b200z_batch_destroy(b200z_batch *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    delete b;
}

// ---------------------------------------------------------------------------------------------------------------
// Pipelined one-shot for HOST buffers: the frame list is cut into a few chunks; while chunk i is being decoded,
// chunk i+1 is planned on the host and its input crosses PCIe, and chunk i-1's plaintext is on its way back.
// Three streams (H2D, compute, D2H) + two descriptor/scratch sets; all device buffers live in the context and are
// reused across calls.
// ---------------------------------------------------------------------------------------------------------------
struct PipeResources {
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    // chunk i's kernels run on stream pair i & 1, so the (latency-bound) kernels of neighbouring chunks overlap
    cudaStream_t k_main[2] = {nullptr, nullptr}, k_side[2] = {nullptr, nullptr};
    cudaEvent_t k_fork[2] = {nullptr, nullptr}, k_join[2] = {nullptr, nullptr};
    b200z_batch *set[2] = {nullptr, nullptr};
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_k[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    FrameState *h_states[2] = {nullptr, nullptr};   // pinned
    size_t h_states_cap[2] = {0, 0};
    DevBuf d_in[2];
    DevBuf d_out;
};

static void pipe_free(b200z_ctx *c) {
    PipeResources *p = c->pipe;
    if (!p) return;
    for (int i = 0; i < 2; i++) {
        if (p->set[i]) delete p->set[i];
        if (p->ev_h2d[i]) cudaEventDestroy(p->ev_h2d[i]);
        if (p->ev_k[i]) cudaEventDestroy(p->ev_k[i]);
        if (p->ev_done[i]) cudaEventDestroy(p->ev_done[i]);
        if (p->k_fork[i]) cudaEventDestroy(p->k_fork[i]);
        if (p->k_join[i]) cudaEventDestroy(p->k_join[i]);
        if (p->k_main[i]) cudaStreamDestroy(p->k_main[i]);
        if (p->k_side[i]) cudaStreamDestroy(p->k_side[i]);
        if (p->h_states[i]) cudaFreeHost(p->h_states[i]);
    }
    if (p->s_h2d) cudaStreamDestroy(p->s_h2d);
    if (p->s_d2h) cudaStreamDestroy(p->s_d2h);
    delete p;
    c->pipe = nullptr;
}

static int pipe_get(b200z_ctx *c, PipeResources **out) {
    if (!c->pipe) {
        std::unique_ptr<PipeResources> p(new PipeResources());
        CU(c, cudaStreamCreateWithFlags(&p->s_h2d, cudaStreamNonBlocking));
        CU(c, cudaStreamCreateWithFlags(&p->s_d2h, cudaStreamNonBlocking));
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        for (int i = 0; i < 2; i++) {
            CU(c, cudaStreamCreateWithPriority(&p->k_main[i], cudaStreamNonBlocking, prio_hi));
            CU(c, cudaStreamCreateWithPriority(&p->k_side[i], cudaStreamNonBlocking, prio_lo));
            CU(c, cudaEventCreateWithFlags(&p->k_fork[i], cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&p->k_join[i], cudaEventDisableTiming));
            p->set[i] = new b200z_batch();
            p->set[i]->ctx = c;
            CU(c, cudaEventCreateWithFlags(&p->ev_h2d[i], cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&p->ev_k[i], cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&p->ev_done[i], cudaEventDisableTiming));
        }
        c->pipe = p.release();
    }
    *out = c->pipe;
    return 0;
}

static int decode_frames_pipelined(b200z_ctx *c, const uint8_t *input, size_t input_len, const b200z_frame_io *frames, size_t nframes,
                                   const b200z_dict *const *dicts, size_t ndicts, const b200z_dict *forced, uint64_t max_window, uint8_t *output,
                                   size_t output_cap, b200z_frame_result *results, size_t nchunks) {
    PipeResources *p = nullptr;
    if (int e = pipe_get(c, &p)) return e;
    if (int e = p->d_out.ensure(output_cap + 64, false)) return e;
    uint8_t *d_out = p->d_out.as<uint8_t>();
    // chunk boundaries: consecutive frames, roughly equal output bytes
    uint64_t total_cap = 0;
    for (size_t i = 0; i < nframes; i++) total_cap += frames[i].out_cap;
    std::vector<size_t> cut(1, 0);
    {
        uint64_t acc = 0, per = total_cap / nchunks + 1;
        for (size_t i = 0; i < nframes; i++) {
            acc += frames[i].out_cap;
            if (acc >= per * cut.size() && i + 1 < nframes && cut.size() < nchunks) cut.push_back(i + 1);
        }
        cut.push_back(nframes);
    }
    const bool trace = getenv("B200Z_TRACE") != nullptr;
    auto t_start = std::chrono::steady_clock::now();
    auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
    struct Pending { size_t f0 = 0, f1 = 0; bool live = false; } pend[2];
    auto retire = [&](int s) -> int {   // results of the chunk that used set s
        if (!pend[s].live) return 0;
        CU(c, cudaEventSynchronize(p->ev_done[s]));
        b200z_batch *b = p->set[s];
        for (size_t i = pend[s].f0; i < pend[s].f1; i++) {
            int32_t sf = b->info[i - pend[s].f0].sub_frame;
            fill_result(b, i - pend[s].f0, sf >= 0 ? &p->h_states[s][sf] : nullptr, results[i]);
        }
        pend[s].live = false;
        return 0;
    };
    for (size_t ci = 0; ci + 1 < cut.size(); ci++) {
        const int s = (int)(ci & 1);
        const size_t f0 = cut[ci], f1 = cut[ci + 1];
        double t0 = now_ms();
        if (int e = retire(s)) return e;
        double t1 = now_ms();
        b200z_batch *b = p->set[s];
        if (int e = plan_batch(b, input, input_len, frames + f0, f1 - f0, dicts, ndicts, forced, max_window)) return e;
        double t2 = now_ms();
        // input byte range and output byte range of this chunk
        uint64_t ilo = UINT64_MAX, ihi = 0, olo = UINT64_MAX, ohi = 0;
        for (size_t i = f0; i < f1; i++) {
            if (frames[i].src_off > input_len || frames[i].src_size > input_len - frames[i].src_off) continue;
            ilo = std::min<uint64_t>(ilo, frames[i].src_off); ihi = std::max<uint64_t>(ihi, frames[i].src_off + frames[i].src_size);
            if (frames[i].out_cap) { olo = std::min<uint64_t>(olo, frames[i].out_off); ohi = std::max<uint64_t>(ohi, frames[i].out_off + frames[i].out_cap); }
        }
        if (ihi < ilo) { ilo = ihi = 0; }
        if (ohi < olo) { olo = ohi = 0; }
        ohi = std::min<uint64_t>(ohi, output_cap); olo = std::min<uint64_t>(olo, ohi);
        if (int e = p->d_in[s].ensure(ihi - ilo + 32)) return e;
        if (ihi > ilo) CU(c, cudaMemcpyAsync(p->d_in[s].p, input + ilo, ihi - ilo, cudaMemcpyHostToDevice, p->s_h2d));
        if (int e = b->sub.upload(c, p->s_h2d)) return e;
        CU(c, cudaEventRecord(p->ev_h2d[s], p->s_h2d));
        cudaStream_t km = p->k_main[s];
        CU(c, cudaStreamWaitEvent(km, p->ev_h2d[s], 0));
        PipelineArgs a = b->sub.args(p->d_in[s].as<uint8_t>() - ilo, d_out, output_cap);
        PipelineStreams ps{km, p->k_side[s], p->k_fork[s], p->k_join[s]};
        int le = launch_pipeline_overlapped(a, ps);
        if (le) return c->set_cuda_err((cudaError_t)le, "launch_pipeline");
        c->launches += pipeline_launch_count(a);
        b->checksummed = false;
        if ((c->flags & B200Z_FLAG_CHECKSUM) && a.nframes) {
            if ((le = launch_checksum(a, km))) return c->set_cuda_err((cudaError_t)le, "launch_checksum");
            c->launches += 1;
            b->checksummed = true;
        }
        CU(c, cudaEventRecord(p->ev_k[s], km));
        CU(c, cudaStreamWaitEvent(p->s_d2h, p->ev_k[s], 0));
        size_t nst = b->sub.states.size();
        if (nst > p->h_states_cap[s]) {
            if (p->h_states[s]) cudaFreeHost(p->h_states[s]);
            p->h_states[s] = nullptr; p->h_states_cap[s] = 0;
            CU(c, cudaMallocHost((void **)&p->h_states[s], (nst + nst / 2 + 16) * sizeof(FrameState)));
            p->h_states_cap[s] = nst + nst / 2 + 16;
        }
        if (nst) CU(c, cudaMemcpyAsync(p->h_states[s], b->sub.d_states.p, nst * sizeof(FrameState), cudaMemcpyDeviceToHost, p->s_d2h));
        if (ohi > olo) CU(c, cudaMemcpyAsync(output + olo, d_out + olo, ohi - olo, cudaMemcpyDeviceToHost, p->s_d2h));
        CU(c, cudaEventRecord(p->ev_done[s], p->s_d2h));
        pend[s].f0 = f0; pend[s].f1 = f1; pend[s].live = true;
        if (trace) fprintf(stderr, "[b200z] chunk %zu frames %zu..%zu: start %.2f retire-wait %.2f plan %.2f enqueue %.2f ms\n", ci, f0, f1, t0, t1 - t0, t2 - t1, now_ms() - t2);
    }
    if (int e = retire(0)) return e;
    if (int e = retire(1)) return e;
    if (trace) fprintf(stderr, "[b200z] pipelined one-shot done at %.2f ms\n", now_ms());
    return 0;
}

extern "C" int b200z_decode_frames_batch(b200z_ctx *c, const uint8_t *input, size_t input_len, int input_mem, const b200z_frame_io *frames,
                                         size_t nframes, const b200z_dict *const *dicts, size_t ndicts, const b200z_dict *forced,
                                         uint64_t max_window, uint8_t *output, size_t output_cap, int output_mem, b200z_frame_result *results) {
    if (!c || !results || (!output && output_cap)) return B200Z_ERR_INVALID_ARGUMENT;
    if (input_mem != B200Z_MEM_DEVICE && output_mem != B200Z_MEM_DEVICE && nframes >= 64) {
        // host in, host out: overlap planning, PCIe and kernels
        if (int e0 = c->use()) return e0;
        if ((!input && input_len) || (!frames && nframes) || (!dicts && ndicts)) return B200Z_ERR_INVALID_ARGUMENT;
        uint64_t total_cap = 0;
        for (size_t i = 0; i < nframes; i++) total_cap += frames[i].out_cap;
        uint64_t chunk_bytes = 256ull << 20;   // ~4 chunks per GiB: PCIe transfers and kernels of neighbouring chunks overlap
        if (const char *ev = getenv("B200Z_PIPELINE_CHUNK_BYTES")) { uint64_t v = strtoull(ev, nullptr, 10); if (v >= 4096) chunk_bytes = v; }
        size_t nchunks = (size_t)std::min<uint64_t>(16, std::max<uint64_t>(1, total_cap / chunk_bytes));
        return decode_frames_pipelined(c, input, input_len, frames, nframes, dicts, ndicts, forced, max_window, output, output_cap, results, nchunks);
    }
    b200z_batch *b = nullptr;
    int e = b200z_batch_prepare(c, input, input_len, input_mem, frames, nframes, dicts, ndicts, forced, max_window, &b);
    if (e) return e;
    std::unique_ptr<b200z_batch, void (*)(b200z_batch *)> guard(b, b200z_batch_destroy);
    DevBuf d_out;
    uint8_t *dout = output;
    if (output_mem != B200Z_MEM_DEVICE) {
        if ((e = d_out.ensure(output_cap + 16, false))) return e;
        dout = d_out.as<uint8_t>();
    }
    if ((e = b200z_batch_run(b, dout, output_cap))) return e;
    if ((e = b200z_batch_finish(b, results))) return e;
    if (output_mem != B200Z_MEM_DEVICE) {
        // one D2H covering every produced byte (frames are normally packed back to back by the caller)
        uint64_t lo = UINT64_MAX, hi = 0;
        for (size_t i = 0; i < nframes; i++)
            if (results[i].out_size) { lo = std::min<uint64_t>(lo, frames[i].out_off); hi = std::max<uint64_t>(hi, frames[i].out_off + results[i].out_size); }
        if (hi > lo) {
            hi = std::min<uint64_t>(hi, output_cap);
            CU(c, cudaMemcpyAsync(output + lo, dout + lo, hi - lo, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
        }
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// tier 1b: block-level batch entry -- replaces the call site of the hot path, BlockDecoder::decompress_block
// (block_decoder.rs:97-197), for a host that keeps the reference's own header parsing.
// ---------------------------------------------------------------------------------------------------------------
extern "C" int b200z_decode_blocks_batch(b200z_ctx *c, const b200z_block_desc *blocks, size_t nblocks, const b200z_block_frame *frames, size_t nframes,
                                         const uint8_t *compressed, size_t compressed_len, int compressed_mem, uint8_t *output, size_t output_cap,
                                         int output_mem, b200z_block_status *status, uint64_t *frame_out_size) {
    if (!c || (!blocks && nblocks) || (!frames && nframes) || (!compressed && compressed_len) || (!output && output_cap)) return B200Z_ERR_INVALID_ARGUMENT;
    if (int e = c->use()) return e;
    std::vector<uint8_t> host_copy;
    const uint8_t *hin = compressed;
    if (compressed_mem == B200Z_MEM_DEVICE) {   // the section headers are walked on the host (as in b200z_batch_prepare)
        host_copy.resize(compressed_len);
        if (compressed_len) CU(c, cudaMemcpy(host_copy.data(), compressed, compressed_len, cudaMemcpyDeviceToHost));
        hin = host_copy.data();
    }
    Submission s;
    std::vector<const b200z_dict *> dlist;
    std::vector<int64_t> sub_of(nblocks, -1);      // caller's block index -> descriptor index in the submission
    std::vector<uint32_t> frame_first(nframes, 0);
    for (size_t f = 0; f < nframes; f++) {
        const b200z_block_frame &bf = frames[f];
        if ((uint64_t)bf.first_block + bf.num_blocks > nblocks) return B200Z_ERR_INVALID_ARGUMENT;
        int dict_idx = -1;
        if (bf.dict) {
            auto it = std::find(dlist.begin(), dlist.end(), bf.dict);
            if (it == dlist.end()) { dlist.push_back(bf.dict); s.carries.push_back(carry_of_dict(bf.dict)); dict_idx = (int)dlist.size() - 1; }
            else dict_idx = (int)(it - dlist.begin());
        }
        FrameDesc fd;
        memset(&fd, 0, sizeof fd);
        fd.out_off = bf.out_off; fd.out_cap = bf.out_cap; fd.window_size = bf.window_size;
        fd.dict = bf.dict ? bf.dict->d_content : nullptr; fd.dict_len = bf.dict ? bf.dict->content_len : 0;
        fd.first_block = (uint32_t)s.descs.size();
        frame_first[f] = fd.first_block;
        FrameState st;
        memset(&st, 0, sizeof st);
        st.hist[0] = bf.dict ? bf.dict->hist[0] : 1; st.hist[1] = bf.dict ? bf.dict->hist[1] : 4; st.hist[2] = bf.dict ? bf.dict->hist[2] : 8;
        TableCursor cur;
        if (dict_idx >= 0) cursor_from_carry(cur, s.carries[dict_idx], (uint32_t)dict_idx);
        for (uint32_t k = 0; k < bf.num_blocks; k++) {
            const b200z_block_desc &bd = blocks[bf.first_block + k];
            if (bd.block_type > BT_COMPRESSED || bd.src_off > compressed_len || bd.content_size > compressed_len - bd.src_off) return B200Z_ERR_INVALID_ARGUMENT;
            BlockDesc d;
            memset(&d, 0, sizeof d);
            BlockRefs r;
            d.src_off = bd.src_off; d.src_size = bd.content_size; d.frame = (uint32_t)f; d.btype = bd.block_type; d.raw_size = bd.decompressed_size;
            d.block_in_frame = k; d.last = bd.last_block;
            if (bd.block_type == BT_COMPRESSED) {
                plan_compressed_block(hin + bd.src_off, bd.content_size, d, r, cur, s.n_huf, s.n_fse, s.lit_bytes, s.nseq);
                // the descriptor says what the caller's parsers found: it must be what the content says
                const bool lit_seen = !(d.host_status && (d.host_status >> 24) == 1 && d.lit_type == 0 && d.regen_size == 0 && d.lit_off == 0);
                if (lit_seen && (d.lit_type != bd.literals_type || d.regen_size != bd.regenerated_size)) return B200Z_ERR_INVALID_ARGUMENT;
                if (!d.host_status && (d.nseq != bd.num_sequences || (d.nseq && d.modes != bd.modes))) return B200Z_ERR_INVALID_ARGUMENT;
            } else if (bd.block_type == BT_RAW ? bd.content_size != bd.decompressed_size : bd.content_size != 1) return B200Z_ERR_INVALID_ARGUMENT;
            sub_of[bf.first_block + k] = (int64_t)s.descs.size();
            s.descs.push_back(d); s.refs.push_back(r);
            if (d.host_status) break;   // decompress_block would have returned here: later blocks of the frame are never reached
        }
        fd.nblocks = (uint32_t)s.descs.size() - fd.first_block;
        s.frames.push_back(fd); s.states.push_back(st);
    }
    DevBuf d_in_own, d_out_own;
    const uint8_t *d_in = compressed;
    if (compressed_mem != B200Z_MEM_DEVICE) {
        if (int e = d_in_own.ensure(compressed_len + 16, false)) return e;
        if (compressed_len) CU(c, cudaMemcpyAsync(d_in_own.p, compressed, compressed_len, cudaMemcpyHostToDevice, c->stream));
        d_in = d_in_own.as<uint8_t>();
    }
    uint8_t *d_out = output;
    if (output_mem != B200Z_MEM_DEVICE) {
        if (int e = d_out_own.ensure(output_cap + 16, false)) return e;
        d_out = d_out_own.as<uint8_t>();
    }
    if (int e = s.upload(c)) return e;
    PipelineArgs a = s.args(d_in, d_out, output_cap);
    PipelineStreams ps{c->stream, c->side, c->ev_fork, c->ev_join};
    if (int le = launch_pipeline_overlapped(a, ps)) return c->set_cuda_err((cudaError_t)le, "launch_pipeline");
    c->launches += pipeline_launch_count(a);
    std::vector<FrameState> st(s.states.size());
    std::vector<BlockAux> aux(s.descs.size());
    if (!st.empty()) CU(c, cudaMemcpyAsync(st.data(), s.d_states.p, st.size() * sizeof(FrameState), cudaMemcpyDeviceToHost, c->stream));
    if (!aux.empty()) CU(c, cudaMemcpyAsync(aux.data(), s.d_aux.p, aux.size() * sizeof(BlockAux), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    uint64_t lo = UINT64_MAX, hi = 0;
    for (size_t f = 0; f < nframes; f++) {
        const b200z_block_frame &bf = frames[f];
        const FrameState &fs = st[f];
        if (frame_out_size) frame_out_size[f] = fs.produced;
        if (fs.produced) { lo = std::min<uint64_t>(lo, bf.out_off); hi = std::max<uint64_t>(hi, bf.out_off + fs.produced); }
        if (!status) continue;
        for (uint32_t k = 0; k < bf.num_blocks; k++) {
            b200z_block_status &o = status[bf.first_block + k];
            memset(&o, 0, sizeof o);
            const int64_t si = sub_of[bf.first_block + k];
            const bool failed_here = fs.status && k == fs.error_block;
            if (si < 0 || (fs.status && k > fs.error_block)) { o.status = B200Z_BLOCK_NOT_REACHED; continue; }
            if (failed_here) { o.status = (int32_t)(fs.status & 0xffffu); o.stage = (int32_t)((fs.status >> 16) & 0xffu); continue; }
            const BlockDesc &d = s.descs[(size_t)si];
            o.out_size = d.btype == BT_COMPRESSED ? aux[(size_t)si].out_size : d.raw_size;
        }
    }
    if (output_mem != B200Z_MEM_DEVICE && hi > lo) {
        hi = std::min<uint64_t>(hi, output_cap);
        if (hi > lo) { CU(c, cudaMemcpyAsync(output + lo, d_out + lo, hi - lo, cudaMemcpyDeviceToHost, c->stream)); CU(c, cudaStreamSynchronize(c->stream)); }
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// tier 2: FrameDecoder mirror (decoding/frame_decoder.rs)
// ---------------------------------------------------------------------------------------------------------------
struct b200z_frame_decoder {
    b200z_ctx *ctx = nullptr;
    uint64_t max_window = B200Z_DEFAULT_MAX_WINDOW_SIZE;
    std::map<uint32_t, b200z_dict *> dicts;           // FrameDecoder.dicts (BTreeMap<u32, Dictionary>), owned
    // FrameDecoderState (frame_decoder.rs:86-94)
    bool has_state = false;
    FrameHeader hdr;
    uint64_t window = 0;
    bool frame_finished = false;
    size_t block_counter = 0;
    uint64_t bytes_read_counter = 0;
    bool has_check_sum = false;
    uint32_t check_sum = 0;
    const b200z_dict *using_dict = nullptr;
    uint32_t skip_len = 0;
    int last_stage = 0;
    std::string err;
    // decode buffer on the device: frame bytes [base, produced) live at d_out[0 .. produced-base); the host has
    // drained everything below `drained` (DecodeBuffer::len() == produced - drained, decode_buffer.rs:58)
    DevBuf d_out;
    uint64_t base = 0, produced = 0, drained = 0;
    FrameState state;                                  // host mirror of the device-side frame state
    XXH64State hash;                                   // decode_buffer.rs:16, fed on drain
    // "current tables" (DecoderScratch.huf/.fse): which kinds exist + persistent device copies
    HufSlot *d_carry_huf = nullptr;
    FseSlot *d_carry_fse = nullptr;
    CarrySet carry;                                    // what the next submission starts from
    Submission sub;
    DevBuf d_input;
    std::vector<uint8_t> staging;                      // bytes of the blocks of the current submission
};

static int fd_fail(b200z_frame_decoder *d, int code, int stage) {
    d->last_stage = stage;
    char buf[160];
    snprintf(buf, sizeof buf, "%s (stage %d)", b200z_error_name(code), stage);
    d->err = buf;
    return code;
}

extern "C" int b200z_frame_decoder_new(b200z_ctx *c, b200z_frame_decoder **out) {
    if (!c || !out) return B200Z_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (int e = c->use()) return e;
    std::unique_ptr<b200z_frame_decoder> d(new b200z_frame_decoder());
    d->ctx = c;
    memset(&d->state, 0, sizeof d->state);
    d->hash.reset();
    CU(c, cudaMalloc((void **)&d->d_carry_huf, sizeof(HufSlot)));
    CU(c, cudaMalloc((void **)&d->d_carry_fse, sizeof(FseSlot)));
    *out = d.release();
    return 0;
}
extern "C" void b200z_frame_decoder_free(b200z_frame_decoder *d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    for (auto &kv : d->dicts) dict_free(kv.second);
    if (d->d_carry_huf) cudaFree(d->d_carry_huf);
    if (d->d_carry_fse) cudaFree(d->d_carry_fse);
    delete d;
}
extern "C" void b200z_frame_decoder_set_max_window_size(b200z_frame_decoder *d, uint64_t n) {
    d->max_window = std::min<uint64_t>(n, (1ull << 41) + 7 * (1ull << 38));
}
extern "C" uint64_t b200z_frame_decoder_max_window_size(const b200z_frame_decoder *d) { return d->max_window; }
extern "C" uint32_t b200z_frame_decoder_skip_frame_length(const b200z_frame_decoder *d) { return d->skip_len; }
extern "C" int b200z_frame_decoder_last_stage(const b200z_frame_decoder *d) { return d->last_stage; }
extern "C" const char *b200z_frame_decoder_last_error_message(const b200z_frame_decoder *d) { return d->err.c_str(); }

static bool read_exact(b200z_read_fn rd, void *user, uint8_t *buf, size_t n) {
    size_t got = 0;
    while (got < n) { long r = rd(user, buf + got, n - got); if (r <= 0) return false; got += (size_t)r; }
    return true;
}

static void fd_apply_dict(b200z_frame_decoder *d, const b200z_dict *dict) {  // DecoderScratch::init_from_dict, scratch.rs:70-78
    d->carry = carry_of_dict(dict);
    d->state.hist[0] = dict->hist[0]; d->state.hist[1] = dict->hist[1]; d->state.hist[2] = dict->hist[2];
    d->using_dict = dict;
}

// reset (frame_decoder.rs:200-221): read the header through the callback exactly like read_frame_header does
extern "C" int b200z_frame_decoder_reset(b200z_frame_decoder *d, b200z_read_fn rd, void *user) {
    if (!d || !rd) return B200Z_ERR_INVALID_ARGUMENT;
    uint8_t buf[32];
    // pull the header piecewise so that no byte beyond it is consumed (frame.rs:6-85)
    size_t have = 0;
    auto need = [&](size_t n) { if (have >= n) return true; if (!read_exact(rd, user, buf + have, n - have)) return false; have = n; return true; };
    FrameHeader h; uint32_t skip = 0; size_t consumed = 0;
    if (!need(4)) return fd_fail(d, B200Z_ERR_MAGIC_NUMBER_READ, B200Z_STAGE_FRAME_HEADER);
    uint32_t magic = (uint32_t)buf[0] | ((uint32_t)buf[1] << 8) | ((uint32_t)buf[2] << 16) | ((uint32_t)buf[3] << 24);
    if (magic >= 0x184D2A50u && magic <= 0x184D2A5Fu) {
        if (!need(8)) return fd_fail(d, B200Z_ERR_FRAME_DESCRIPTOR_READ, B200Z_STAGE_FRAME_HEADER);
        parse_frame_header(buf, 8, h, skip, consumed);
        d->skip_len = skip;
        return fd_fail(d, B200Z_ERR_SKIP_FRAME, B200Z_STAGE_FRAME_HEADER);
    }
    if (magic != 0xFD2FB528u) return fd_fail(d, B200Z_ERR_BAD_MAGIC_NUMBER, B200Z_STAGE_FRAME_HEADER);
    if (!need(5)) return fd_fail(d, B200Z_ERR_FRAME_DESCRIPTOR_READ, B200Z_STAGE_FRAME_HEADER);
    uint8_t desc = buf[4];
    size_t pos = 5;
    bool single = (desc >> 5) & 1;
    if (!single) { if (!need(pos + 1)) return fd_fail(d, B200Z_ERR_WINDOW_DESCRIPTOR_READ, B200Z_STAGE_FRAME_HEADER); pos += 1; }
    static const uint8_t did_len[4] = {0, 1, 2, 4};
    size_t dl = did_len[desc & 3];
    if (dl) { if (!need(pos + dl)) return fd_fail(d, B200Z_ERR_DICTIONARY_ID_READ, B200Z_STAGE_FRAME_HEADER); pos += dl; }
    uint32_t flag = desc >> 6;
    size_t fl = flag == 0 ? (single ? 1 : 0) : (flag == 1 ? 2 : (flag == 2 ? 4 : 8));
    if (fl) { if (!need(pos + fl)) return fd_fail(d, B200Z_ERR_FRAME_CONTENT_SIZE_READ, B200Z_STAGE_FRAME_HEADER); pos += fl; }
    int e = parse_frame_header(buf, pos, h, skip, consumed);
    if (e) return fd_fail(d, e, B200Z_STAGE_FRAME_HEADER);
    uint64_t window = 0;
    if ((e = frame_window_size(h, window))) return fd_fail(d, e, B200Z_STAGE_FRAME_HEADER);
    if (window > d->max_window) return fd_fail(d, B200Z_ERR_WINDOW_SIZE_TOO_BIG, B200Z_STAGE_FRAME_HEADER);
    // FrameDecoderState::new / reset (:103-134)
    d->hdr = h; d->window = window; d->frame_finished = false; d->block_counter = 0;
    d->bytes_read_counter = h.header_size; d->has_check_sum = false; d->using_dict = nullptr;
    d->base = d->produced = d->drained = 0;
    memset(&d->state, 0, sizeof d->state);
    d->state.hist[0] = 1; d->state.hist[1] = 4; d->state.hist[2] = 8;
    d->hash.reset();
    d->carry = CarrySet();
    d->has_state = true;
    if (h.has_dict_id) {
        auto it = d->dicts.find(h.dict_id);
        if (it == d->dicts.end()) return fd_fail(d, B200Z_ERR_DICT_NOT_PROVIDED, B200Z_STAGE_FRAME_HEADER);
        fd_apply_dict(d, it->second);
    }
    d->last_stage = 0;
    return 0;
}
extern "C" int b200z_frame_decoder_init(b200z_frame_decoder *d, b200z_read_fn rd, void *user) { return b200z_frame_decoder_reset(d, rd, user); }

extern "C" int b200z_frame_decoder_add_dict(b200z_frame_decoder *d, const uint8_t *raw, size_t len) {
    if (!d) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_dict *x = nullptr;
    int e = b200z_dict_create(d->ctx, raw, len, &x);
    if (e) return fd_fail(d, e, B200Z_STAGE_DICTIONARY);
    auto it = d->dicts.find(x->id);
    if (it != d->dicts.end()) { if (d->using_dict == it->second) d->using_dict = nullptr; dict_free(it->second); it->second = x; } else d->dicts[x->id] = x;
    return 0;
}
extern "C" int b200z_frame_decoder_add_raw_content_dict(b200z_frame_decoder *d, uint32_t id, const uint8_t *content, size_t len) {
    if (!d) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_dict *x = nullptr;
    int e = b200z_dict_create_raw_content(d->ctx, id, content, len, &x);
    if (e) return fd_fail(d, e, B200Z_STAGE_DICTIONARY);
    auto it = d->dicts.find(id);
    if (it != d->dicts.end()) { if (d->using_dict == it->second) d->using_dict = nullptr; dict_free(it->second); it->second = x; } else d->dicts[id] = x;
    return 0;
}
extern "C" int b200z_frame_decoder_force_dict(b200z_frame_decoder *d, uint32_t dict_id) {  // :229-243
    if (!d) return B200Z_ERR_INVALID_ARGUMENT;
    if (!d->has_state) return fd_fail(d, B200Z_ERR_NOT_YET_INITIALIZED, 0);
    auto it = d->dicts.find(dict_id);
    if (it == d->dicts.end()) return fd_fail(d, B200Z_ERR_DICT_NOT_PROVIDED, 0);
    fd_apply_dict(d, it->second);
    return 0;
}

static size_t fd_buffer_len(const b200z_frame_decoder *d) { return (size_t)(d->produced - d->drained); }
static bool fd_finished(const b200z_frame_decoder *d) {  // is_finished :284-294
    if (!d->has_state) return true;
    if (d->hdr.content_checksum()) return d->frame_finished && d->has_check_sum;
    return d->frame_finished;
}
static size_t fd_can_drain_to_window(const b200z_frame_decoder *d) {  // decode_buffer.rs:182-188
    size_t n = fd_buffer_len(d);
    return n > d->window ? (size_t)(n - d->window) : 0;
}

// make room for `extra` more bytes behind `produced`, dropping drained bytes when that frees enough
static int fd_reserve_out(b200z_frame_decoder *d, uint64_t extra) {
    b200z_ctx *c = d->ctx;
    uint64_t live = d->produced - d->drained;
    uint64_t need = (d->produced - d->base) + extra + 64;
    if (need <= d->d_out.cap) return 0;
    uint64_t want = std::max<uint64_t>(live + extra + 64, (uint64_t)d->d_out.cap + d->d_out.cap / 2);
    want = std::max<uint64_t>(want, 1u << 20);
    void *np = nullptr;
    if (cudaMalloc(&np, want) != cudaSuccess) { cudaGetLastError(); return B200Z_ERR_OUT_OF_MEMORY; }
    if (live) {
        cudaError_t ce = cudaMemcpyAsync(np, d->d_out.as<uint8_t>() + (d->drained - d->base), live, cudaMemcpyDeviceToDevice, c->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->stream);
        if (ce != cudaSuccess) { cudaFree(np); return c->set_cuda_err(ce, "grow output"); }
    }
    d->d_out.release();
    d->d_out.p = np; d->d_out.cap = want;
    d->base = d->drained;
    return 0;
}

// Decode the blocks gathered in d->sub / d->staging on the GPU; updates produced/state/carry tables.
// Returns 0 or the error of the first failing block (in which case *failed_block is its index in the submission).
static int fd_submit(b200z_frame_decoder *d, const TableCursor &cur, uint32_t *failed_block, uint32_t *done_blocks) {
    b200z_ctx *c = d->ctx;
    Submission &s = d->sub;
    if (int e = c->use()) return e;
    int e;
    if ((e = d->d_input.ensure(d->staging.size() + 16))) return e;
    CU(c, cudaMemcpyAsync(d->d_input.p, d->staging.data(), d->staging.size(), cudaMemcpyHostToDevice, c->stream));
    FrameDesc fd;
    memset(&fd, 0, sizeof fd);
    fd.out_off = 0; fd.window_size = d->window;
    fd.dict = d->using_dict ? d->using_dict->d_content : nullptr; fd.dict_len = d->using_dict ? d->using_dict->content_len : 0;
    fd.first_block = 0; fd.nblocks = (uint32_t)s.descs.size();
    d->state.produced = d->produced; d->state.drained = d->drained; d->state.blocks_done = 0; d->state.status = 0;
    s.frames.assign(1, fd); s.states.assign(1, d->state);
    s.carries.assign(1, d->carry);
    if ((e = s.upload(c))) return e;
    // stage A: tables + literals + sequences; sizes come back so the output can grow before execution
    PipelineArgs a = s.args(d->d_input.as<uint8_t>(), nullptr, 0);
    PipelineArgs a_dec = a; a_dec.nframes = 0;
    int le = launch_pipeline(a_dec, c->stream);
    if (le) return c->set_cuda_err((cudaError_t)le, "launch decode");
    c->launches += pipeline_launch_count(a_dec);
    std::vector<BlockAux> aux(s.descs.size());
    CU(c, cudaMemcpyAsync(aux.data(), s.d_aux.p, aux.size() * sizeof(BlockAux), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    uint64_t extra = 0;
    for (size_t i = 0; i < aux.size(); i++) {   // blocks after the first failing one are never executed (nor looked at by the reference)
        if (s.descs[i].host_status || aux[i].status || aux[i].pad) break;
        extra += aux[i].out_size;
    }
    if ((e = fd_reserve_out(d, extra))) return e;
    // stage B: execution into the persistent window buffer (frame byte 0 sits at d_out - base)
    s.frames[0].out_cap = d->base + d->d_out.cap;
    CU(c, cudaMemcpyAsync(s.d_frames.p, s.frames.data(), sizeof(FrameDesc), cudaMemcpyHostToDevice, c->stream));
    PipelineArgs a_ex = a; a_ex.nblocks = 0;
    a_ex.output = d->d_out.as<uint8_t>() - d->base; a_ex.output_cap = d->base + d->d_out.cap;
    le = launch_pipeline(a_ex, c->stream);
    if (le) return c->set_cuda_err((cudaError_t)le, "launch exec");
    c->launches += pipeline_launch_count(a_ex);
    // carry the current tables over to the next submission (device-to-device, tables never visit the host)
    CarrySet next;
    if (cur.huf.kind == TabRef::SLOT) {
        CU(c, cudaMemcpyAsync(d->d_carry_huf, s.d_huf.as<HufSlot>() + cur.huf.idx, sizeof(HufSlot), cudaMemcpyDeviceToDevice, c->stream));
        next.huf = d->d_carry_huf;
    } else if (cur.huf.kind == TabRef::CARRY) next.huf = d->carry.huf;
    auto carry_fse = [&](const TabRef &t, int which, FseTab *dst, const FseTab *old) -> const FseTab * {
        const FseTab *src = nullptr;
        if (t.kind == TabRef::SLOT) { const FseSlot *sl = s.d_fse.as<FseSlot>() + t.idx; src = which == 0 ? &sl->ll : (which == 1 ? &sl->of : &sl->ml); }
        else if (t.kind == TabRef::PREDEF) { const FseSlot *sl = c->d_predef; return which == 0 ? &sl->ll : (which == 1 ? &sl->of : &sl->ml); }
        else if (t.kind == TabRef::CARRY) return old;
        else return nullptr;
        if (cudaMemcpyAsync(dst, src, sizeof(FseTab), cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess) return nullptr;
        return dst;
    };
    next.ll = carry_fse(cur.ll, 0, &d->d_carry_fse->ll, d->carry.ll);
    next.of = carry_fse(cur.of, 1, &d->d_carry_fse->of, d->carry.of);
    next.ml = carry_fse(cur.ml, 2, &d->d_carry_fse->ml, d->carry.ml);
    FrameState st;
    CU(c, cudaMemcpyAsync(&st, s.d_states.p, sizeof(FrameState), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    d->carry = next;
    d->state = st;
    d->produced = st.produced;
    *done_blocks = st.blocks_done;
    if (st.status) { *failed_block = st.blocks_done; d->last_stage = (int)((st.status >> 16) & 0xff); return (int)(st.status & 0xffff); }
    return 0;
}

namespace {
struct SliceReader { const uint8_t *p; size_t len; };
long slice_read(void *user, uint8_t *buf, size_t n) {  // impl Read for &[u8]
    SliceReader *s = (SliceReader *)user;
    size_t k = std::min(n, s->len);
    if (k) memcpy(buf, s->p, k);
    s->p += k; s->len -= k;
    return (long)k;
}
}  // namespace

// decode_blocks (frame_decoder.rs:309-377).  `slice` != null selects decode_from_to's trailer rule (:505-516):
// the checksum is taken only if its 4 bytes are present, otherwise left for the next call.
static int fd_decode_blocks_impl(b200z_frame_decoder *d, b200z_read_fn rd, void *user, int strategy, size_t n, int *finished, SliceReader *slice) {
    if (!d || !rd) return B200Z_ERR_INVALID_ARGUMENT;
    if (!d->has_state) return fd_fail(d, B200Z_ERR_NOT_YET_INITIALIZED, 0);
    if (d->state.status) return fd_fail(d, (int)(d->state.status & 0xffff), (int)((d->state.status >> 16) & 0xff));
    const size_t buffer_size_before = fd_buffer_len(d);
    const size_t block_counter_before = d->block_counter;
    bool stop = false;
    while (!stop) {
        // gather blocks for one GPU submission.  All / UptoBlocks know where to stop from the headers alone;
        // UptoBytes must see each block's decoded size, so it submits block by block.
        Submission &s = d->sub;
        s.clear();
        d->staging.clear();
        TableCursor cur;
        cursor_from_carry(cur, d->carry, 0);
        std::vector<uint64_t> bytes_after;  // bytes_read_counter after each gathered block
        int pending_err = 0, pending_stage = 0;
        bool saw_last = false;
        uint64_t brc = d->bytes_read_counter;
        size_t gathered_target = strategy == B200Z_STRATEGY_UPTO_BYTES ? 1 : (strategy == B200Z_STRATEGY_UPTO_BLOCKS ? std::max<size_t>(n, 1) - (d->block_counter - block_counter_before) : SIZE_MAX);
        if (strategy == B200Z_STRATEGY_ALL) gathered_target = 4096;  // bound the staging buffer; loop continues
        while (s.descs.size() < gathered_target) {
            uint8_t hb[3];
            if (!read_exact(rd, user, hb, 3)) { pending_err = B200Z_ERR_BLOCK_HEADER_READ; pending_stage = B200Z_STAGE_BLOCK_HEADER; break; }
            BlockHeader bh;
            int e = parse_block_header(hb, bh);
            if (e) { pending_err = e; pending_stage = B200Z_STAGE_BLOCK_HEADER; break; }
            brc += 3;
            size_t off = d->staging.size();
            d->staging.resize(off + bh.content_size);
            if (!read_exact(rd, user, d->staging.data() + off, bh.content_size)) {
                d->staging.resize(off);
                pending_err = bh.type == BT_COMPRESSED ? B200Z_ERR_BLOCK_CONTENT_READ : B200Z_ERR_BLOCK_BODY_READ; pending_stage = B200Z_STAGE_BLOCK_BODY;
                break;
            }
            BlockDesc bd;
            memset(&bd, 0, sizeof bd);
            BlockRefs r;
            bd.src_off = off; bd.src_size = bh.content_size; bd.frame = 0; bd.btype = bh.type; bd.raw_size = bh.decompressed_size;
            bd.block_in_frame = (uint32_t)(d->block_counter + s.descs.size()); bd.last = bh.last;
            if (bh.type == BT_COMPRESSED) plan_compressed_block(d->staging.data() + off, bh.content_size, bd, r, cur, s.n_huf, s.n_fse, s.lit_bytes, s.nseq);
            s.descs.push_back(bd); s.refs.push_back(r);
            brc += bh.content_size;
            bytes_after.push_back(brc);
            if (bd.host_status) break;
            if (bh.last) { saw_last = true; break; }
        }
        uint32_t failed = 0, done = 0;
        int e = 0;
        if (!s.descs.empty()) e = fd_submit(d, cur, &failed, &done);
        // counters exactly as the reference leaves them (:325-343)
        if (done > 0) d->bytes_read_counter = bytes_after[done - 1];
        d->block_counter += done;
        if (e) {
            if (d->last_stage >= B200Z_STAGE_BLOCK_BODY && d->last_stage <= B200Z_STAGE_EXECUTE) d->bytes_read_counter += 3;
            return fd_fail(d, e, d->last_stage);
        }
        if (pending_err) {
            if (pending_stage == B200Z_STAGE_BLOCK_BODY) d->bytes_read_counter += 3;
            d->state.status = mk_status((uint32_t)pending_err, (uint32_t)pending_stage);
            return fd_fail(d, pending_err, pending_stage);
        }
        if (saw_last) {
            d->frame_finished = true;
            if (d->hdr.content_checksum() && !(slice && slice->len < 4)) {
                uint8_t cs[4];
                if (!read_exact(rd, user, cs, 4)) return fd_fail(d, B200Z_ERR_FAILED_TO_READ_CHECKSUM, B200Z_STAGE_CHECKSUM);
                d->bytes_read_counter += 4;
                d->check_sum = (uint32_t)cs[0] | ((uint32_t)cs[1] << 8) | ((uint32_t)cs[2] << 16) | ((uint32_t)cs[3] << 24);
                d->has_check_sum = true;
            }
            break;
        }
        if (strategy == B200Z_STRATEGY_UPTO_BLOCKS) stop = d->block_counter - block_counter_before >= n;
        else if (strategy == B200Z_STRATEGY_UPTO_BYTES) stop = fd_buffer_len(d) - buffer_size_before >= n;
    }
    d->last_stage = 0;
    if (finished) *finished = d->frame_finished ? 1 : 0;
    return 0;
}

extern "C" int b200z_frame_decoder_decode_blocks(b200z_frame_decoder *d, b200z_read_fn rd, void *user, int strategy, size_t n, int *finished) {
    return fd_decode_blocks_impl(d, rd, user, strategy, n, finished, nullptr);
}

// drain `amount` bytes from the front of the device buffer into host memory / a writer; feeds the hash
static long fd_drain(b200z_frame_decoder *d, size_t amount, uint8_t *target, b200z_write_fn wr, void *user) {
    if (amount == 0) return 0;
    b200z_ctx *c = d->ctx;
    if (c->use()) return -1;
    std::vector<uint8_t> tmp;
    uint8_t *dst = target;
    if (!dst) { tmp.resize(amount); dst = tmp.data(); }
    if (cudaMemcpyAsync(dst, d->d_out.as<uint8_t>() + (d->drained - d->base), amount, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); return -1; }
    size_t written = amount;
    bool failed = false;
    if (!target) {  // write_all_bytes (decode_buffer.rs:318-328)
        written = 0;
        while (written < amount) {
            long w = wr(user, dst + written, amount - written);
            if (w == 0) break;
            if (w < 0) { failed = true; break; }
            written += (size_t)w;
        }
    }
    d->hash.update(dst, written);
    d->drained += written;
    return failed ? -1 : (long)written;
}

extern "C" long b200z_frame_decoder_read(b200z_frame_decoder *d, uint8_t *buf, size_t len) {  // impl Read :615-627
    if (!d || !d->has_state) return 0;
    size_t amount = d->frame_finished ? std::min(len, fd_buffer_len(d)) : std::min(len, fd_can_drain_to_window(d));
    return fd_drain(d, amount, buf, nullptr, nullptr);
}
extern "C" long b200z_frame_decoder_collect_to_writer(b200z_frame_decoder *d, b200z_write_fn wr, void *user) {  // :393-404
    if (!d || !d->has_state || !wr) return 0;
    size_t amount = fd_finished(d) ? fd_buffer_len(d) : fd_can_drain_to_window(d);
    return fd_drain(d, amount, nullptr, wr, user);
}
extern "C" size_t b200z_frame_decoder_can_collect(const b200z_frame_decoder *d) {  // :409-424
    if (!d || !d->has_state) return 0;
    return fd_finished(d) ? fd_buffer_len(d) : fd_can_drain_to_window(d);
}
extern "C" int b200z_frame_decoder_is_finished(const b200z_frame_decoder *d) { return d ? fd_finished(d) : 1; }
extern "C" size_t b200z_frame_decoder_blocks_decoded(const b200z_frame_decoder *d) { return d && d->has_state ? d->block_counter : 0; }
extern "C" uint64_t b200z_frame_decoder_bytes_read_from_source(const b200z_frame_decoder *d) { return d && d->has_state ? d->bytes_read_counter : 0; }
extern "C" uint64_t b200z_frame_decoder_content_size(const b200z_frame_decoder *d) { return d && d->has_state ? d->hdr.frame_content_size : 0; }
extern "C" int b200z_frame_decoder_get_checksum_from_data(const b200z_frame_decoder *d, uint32_t *out) {
    if (!d || !d->has_state || !d->has_check_sum) return 0;
    *out = d->check_sum; return 1;
}
extern "C" int b200z_frame_decoder_get_calculated_checksum(const b200z_frame_decoder *d, uint32_t *out) {
    if (!d || !d->has_state) return 0;
    *out = (uint32_t)d->hash.digest(); return 1;
}

// decode_from_to (frame_decoder.rs:439-529): decodes as many WHOLE blocks as `src` holds
extern "C" int b200z_frame_decoder_decode_from_to(b200z_frame_decoder *d, const uint8_t *src, size_t src_len, uint8_t *dst, size_t dst_len,
                                                  size_t *read, size_t *written) {
    if (!d || !read || !written) return B200Z_ERR_INVALID_ARGUMENT;
    uint64_t at_start = d->has_state ? d->bytes_read_counter : 0;
    if (!fd_finished(d) || !d->has_state) {
        SliceReader mt{src, src_len};
        if (!d->has_state) { int e = b200z_frame_decoder_init(d, slice_read, &mt); if (e) return e; }
        if (d->hdr.content_checksum() && d->frame_finished && !d->has_check_sum) {  // :465-477
            if (mt.len >= 4) {
                d->bytes_read_counter += 4;
                d->check_sum = (uint32_t)mt.p[0] | ((uint32_t)mt.p[1] << 8) | ((uint32_t)mt.p[2] << 16) | ((uint32_t)mt.p[3] << 24);
                d->has_check_sum = true;
            }
            *read = 4; *written = 0;
            return 0;
        }
        // the reference loops block by block while a whole block is present (:479-518); count them from the
        // headers, then decode exactly those in one submission
        size_t k = 0;
        int hdr_err = 0;
        {
            SliceReader probe = mt;
            while (probe.len >= 3) {
                BlockHeader bh;
                int e = parse_block_header(probe.p, bh);
                if (e) { hdr_err = e; break; }
                if (probe.len - 3 < bh.content_size) break;
                probe.p += 3 + bh.content_size; probe.len -= 3 + bh.content_size;
                k++;
                if (bh.last) break;
            }
        }
        if (k > 0) {
            int e = fd_decode_blocks_impl(d, slice_read, &mt, B200Z_STRATEGY_UPTO_BLOCKS, k, nullptr, &mt);
            if (e) return e;
        }
        if (hdr_err && !d->frame_finished) return fd_fail(d, hdr_err, B200Z_STAGE_BLOCK_HEADER);
    }
    long r = b200z_frame_decoder_read(d, dst, dst_len);
    if (r < 0) return fd_fail(d, B200Z_ERR_FAILED_TO_DRAIN_DECODEBUFFER, B200Z_STAGE_DRAIN);
    *written = (size_t)r;
    *read = (size_t)(d->bytes_read_counter - at_start);
    return 0;
}

// decode_all (frame_decoder.rs:541-577)
extern "C" int b200z_frame_decoder_decode_all(b200z_frame_decoder *d, const uint8_t *input, size_t input_len, uint8_t *output, size_t output_cap, size_t *written) {
    if (!d || !written) return B200Z_ERR_INVALID_ARGUMENT;
    SliceReader in{input, input_len};
    size_t total = 0;
    while (in.len != 0) {
        int e = b200z_frame_decoder_init(d, slice_read, &in);
        if (e == B200Z_ERR_SKIP_FRAME) {
            if ((size_t)d->skip_len > in.len) return fd_fail(d, B200Z_ERR_FAILED_TO_SKIP_FRAME, 0);
            in.p += d->skip_len; in.len -= d->skip_len;
            continue;
        }
        if (e) return e;
        for (;;) {
            if ((e = b200z_frame_decoder_decode_blocks(d, slice_read, &in, B200Z_STRATEGY_UPTO_BYTES, 1024 * 1024, nullptr))) return e;
            long w = b200z_frame_decoder_read(d, output + total, output_cap - total);
            if (w < 0) return fd_fail(d, B200Z_ERR_FAILED_TO_DRAIN_DECODEBUFFER, B200Z_STAGE_DRAIN);
            total += (size_t)w;
            if (b200z_frame_decoder_can_collect(d) != 0) return fd_fail(d, B200Z_ERR_TARGET_TOO_SMALL, 0);
            if (fd_finished(d)) break;
        }
    }
    *written = total;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// StreamingDecoder mirror (decoding/streaming_decoder.rs)
// ---------------------------------------------------------------------------------------------------------------
struct b200z_streaming_decoder {
    b200z_frame_decoder *dec = nullptr;
    bool owns = false;
    b200z_read_fn rd = nullptr;
    void *user = nullptr;
};

static int sd_make(b200z_frame_decoder *dec, bool owns, b200z_read_fn rd, void *user, b200z_streaming_decoder **out) {
    int e = b200z_frame_decoder_init(dec, rd, user);
    if (e) { if (owns) b200z_frame_decoder_free(dec); return e; }
    b200z_streaming_decoder *s = new b200z_streaming_decoder();
    s->dec = dec; s->owns = owns; s->rd = rd; s->user = user;
    *out = s;
    return 0;
}
extern "C" int b200z_streaming_decoder_new(b200z_ctx *c, b200z_read_fn rd, void *user, b200z_streaming_decoder **out) {
    if (!c || !rd || !out) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_frame_decoder *dec = nullptr;
    int e = b200z_frame_decoder_new(c, &dec);
    if (e) return e;
    return sd_make(dec, true, rd, user, out);
}
extern "C" int b200z_streaming_decoder_new_with_decoder(b200z_read_fn rd, void *user, b200z_frame_decoder *dec, b200z_streaming_decoder **out) {
    if (!dec || !rd || !out) return B200Z_ERR_INVALID_ARGUMENT;
    return sd_make(dec, false, rd, user, out);
}
extern "C" int b200z_streaming_decoder_new_with_max_window_size(b200z_ctx *c, b200z_read_fn rd, void *user, uint64_t mw, b200z_streaming_decoder **out) {
    if (!c || !rd || !out) return B200Z_ERR_INVALID_ARGUMENT;
    b200z_frame_decoder *dec = nullptr;
    int e = b200z_frame_decoder_new(c, &dec);
    if (e) return e;
    b200z_frame_decoder_set_max_window_size(dec, mw);
    return sd_make(dec, true, rd, user, out);
}
extern "C" long b200z_streaming_decoder_read(b200z_streaming_decoder *s, uint8_t *buf, size_t len, int *error) {  // :118-155
    if (error) *error = 0;
    if (!s) return -1;
    b200z_frame_decoder *d = s->dec;
    if (fd_finished(d) && b200z_frame_decoder_can_collect(d) == 0) return 0;
    while (b200z_frame_decoder_can_collect(d) < len && !fd_finished(d)) {
        size_t need = len - b200z_frame_decoder_can_collect(d);
        int e = b200z_frame_decoder_decode_blocks(d, s->rd, s->user, B200Z_STRATEGY_UPTO_BYTES, need, nullptr);
        if (e) { if (error) *error = e; return -1; }
    }
    return b200z_frame_decoder_read(d, buf, len);
}
extern "C" b200z_frame_decoder *b200z_streaming_decoder_frame_decoder(b200z_streaming_decoder *s) { return s ? s->dec : nullptr; }
extern "C" b200z_frame_decoder *b200z_streaming_decoder_into_frame_decoder(b200z_streaming_decoder *s) {
    if (!s) return nullptr;
    b200z_frame_decoder *d = s->dec;
    delete s;
    return d;
}
extern "C" void b200z_streaming_decoder_free(b200z_streaming_decoder *s) {
    if (!s) return;
    if (s->owns) b200z_frame_decoder_free(s->dec);
    delete s;
}

// ---------------------------------------------------------------------------------------------------------------
// compression (compress.cu): the plan is block counts and scratch offsets; scratch is a fixed worst case per block, kept in
// the context and reused across calls.
// ---------------------------------------------------------------------------------------------------------------
struct CompressResources {
    DevBuf d_in, d_out, d_frames, d_blocks, d_bout, d_block_off, d_hash, d_results, d_lits, d_seqs, d_body, d_cand;
};
static void comp_free(b200z_ctx *c) { delete c->comp; c->comp = nullptr; }

extern "C" size_t b200z_compress_bound(size_t n) {
    return 6 + enc_fcs_bytes(n) + 3 * (size_t)enc_num_blocks(n) + n + 4;
}

extern "C" int b200z_compress_frames_batch(b200z_ctx *c, const uint8_t *input, size_t input_len, int input_mem, const b200z_frame_io *frames,
                                           size_t nframes, int level, uint32_t flags, uint8_t *output, size_t output_cap, int output_mem,
                                           b200z_compress_result *results) {
    if (level >= B200Z_LEVEL_DEFAULT && level <= B200Z_LEVEL_BEST) return B200Z_ERR_REFERENCE_WOULD_PANIC;   // unimplemented!()
    if (level != B200Z_LEVEL_UNCOMPRESSED && level != B200Z_LEVEL_FASTEST) return B200Z_ERR_INVALID_ARGUMENT;
    if (!c || (flags & ~(B200Z_COMPRESS_CHECKSUM | B200Z_COMPRESS_CONTENT_SIZE)) || (!results && nframes) || (!frames && nframes) ||
        (!input && input_len) || (!output && output_cap))
        return B200Z_ERR_INVALID_ARGUMENT;
    if (int e = c->use()) return e;
    if (!nframes) return 0;
    std::vector<CFrame> hf(nframes);
    std::vector<CBlock> hb;
    uint64_t in_lo = UINT64_MAX, in_hi = 0;
    for (size_t i = 0; i < nframes; i++) {
        const b200z_frame_io &io = frames[i];
        if (io.src_off > input_len || io.src_size > input_len - io.src_off) return B200Z_ERR_INVALID_ARGUMENT;
        const uint64_t nb = enc_num_blocks(io.src_size);
        if (hb.size() + nb > UINT32_MAX) return B200Z_ERR_INVALID_ARGUMENT;
        hf[i] = CFrame{io.src_off, io.src_size, io.out_off, io.out_cap, (uint32_t)hb.size(), (uint32_t)nb};
        for (uint64_t k = 0; k < nb; k++) {
            const uint64_t off = k * ENC_BLOCK;
            hb.push_back(CBlock{io.src_off + off, (uint32_t)std::min<uint64_t>(ENC_BLOCK, io.src_size - off), (uint32_t)i, (uint32_t)(k + 1 == nb), 0});
        }
        in_lo = std::min<uint64_t>(in_lo, io.src_off); in_hi = std::max<uint64_t>(in_hi, io.src_off + io.src_size);
    }
    if (!c->comp) c->comp = new CompressResources();
    CompressResources &R = *c->comp;
    const size_t nblocks = hb.size();
    const uint32_t match_ctas = c->match_ctas;
    int e = 0;
    if ((e = R.d_frames.ensure(nframes * sizeof(CFrame))) || (e = R.d_blocks.ensure(nblocks * sizeof(CBlock))) ||
        (e = R.d_bout.ensure(nblocks * sizeof(CBlockOut))) || (e = R.d_block_off.ensure(nblocks * 8)) || (e = R.d_hash.ensure(nframes * 8)) ||
        (e = R.d_results.ensure(nframes * sizeof(b200z_compress_result))))
        return e;
    if (level == B200Z_LEVEL_FASTEST &&
        ((e = R.d_lits.ensure(nblocks * (size_t)ENC_BLOCK)) || (e = R.d_seqs.ensure(nblocks * (size_t)ENC_MAX_SEQ * sizeof(EncSeq))) ||
         (e = R.d_body.ensure(nblocks * (size_t)ENC_BODY_STRIDE)) || (e = R.d_cand.ensure((size_t)match_ctas * ENC_BLOCK * 4))))
        return e;
    const uint8_t *d_in = input;
    if (input_mem != B200Z_MEM_DEVICE) {
        if ((e = R.d_in.ensure(in_hi > in_lo ? in_hi - in_lo + 16 : 16))) return e;
        if (in_hi > in_lo) CU(c, cudaMemcpyAsync(R.d_in.p, input + in_lo, in_hi - in_lo, cudaMemcpyHostToDevice, c->stream));
        d_in = R.d_in.as<uint8_t>() - (in_hi > in_lo ? in_lo : 0);
    }
    uint8_t *d_out = output;
    if (output_mem != B200Z_MEM_DEVICE) {
        if ((e = R.d_out.ensure(output_cap + 16))) return e;
        d_out = R.d_out.as<uint8_t>();
    }
    CU(c, cudaMemcpyAsync(R.d_frames.p, hf.data(), nframes * sizeof(CFrame), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(R.d_blocks.p, hb.data(), nblocks * sizeof(CBlock), cudaMemcpyHostToDevice, c->stream));
    CompressArgs a{d_in, d_out, output_cap, R.d_frames.as<CFrame>(), R.d_blocks.as<CBlock>(), R.d_bout.as<CBlockOut>(), R.d_block_off.as<uint64_t>(),
                   R.d_hash.as<uint64_t>(), R.d_results.as<b200z_compress_result>(), R.d_lits.as<uint8_t>(), R.d_seqs.as<EncSeq>(), R.d_body.as<uint8_t>(),
                   R.d_cand.as<uint32_t>(), (uint32_t)nblocks, (uint32_t)nframes, (uint32_t)level, flags, match_ctas};
    for (int k = 0; k < kCompressKernels; k++)
        if (int le = launch_compress_stage(a, k, c->stream)) return c->set_cuda_err((cudaError_t)le, kCompressKernelNames[k]);
    c->launches += compress_launch_count(a);
    CU(c, cudaMemcpyAsync(results, R.d_results.p, nframes * sizeof(b200z_compress_result), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (output_mem != B200Z_MEM_DEVICE) {
        // exactly the bytes each frame wrote: the caller's buffer between frames and under failed frames is left alone.  Frames
        // that follow each other without a gap go back in one copy.
        uint64_t lo = 0, hi = 0;
        for (size_t i = 0; i <= nframes; i++) {
            const bool wrote = i < nframes && results[i].status == 0 && results[i].out_size;
            if (wrote && hi > lo && frames[i].out_off == hi) { hi += results[i].out_size; continue; }
            if (hi > lo) CU(c, cudaMemcpyAsync(output + lo, d_out + lo, hi - lo, cudaMemcpyDeviceToHost, c->stream));
            lo = hi = 0;
            if (wrote) { lo = frames[i].out_off; hi = lo + results[i].out_size; }
        }
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return 0;
}

extern "C" int b200z_compress(b200z_ctx *c, b200z_read_fn rd, void *ruser, b200z_write_fn wr, void *wuser, int level, uint32_t flags) {
    if (level >= B200Z_LEVEL_DEFAULT && level <= B200Z_LEVEL_BEST) return B200Z_ERR_REFERENCE_WOULD_PANIC;
    if (!c || !rd || !wr) return B200Z_ERR_INVALID_ARGUMENT;
    std::vector<uint8_t> src;
    for (;;) {   // read to EOF (frame_compressor.rs:151-163)
        const size_t at = src.size();
        src.resize(at + (1u << 20));
        const long r = rd(ruser, src.data() + at, 1u << 20);
        if (r < 0) { src.resize(at); c->err = "read callback failed"; return B200Z_ERR_INVALID_ARGUMENT; }
        src.resize(at + (size_t)r);
        if (r == 0) break;
    }
    const size_t cap = b200z_compress_bound(src.size());
    std::vector<uint8_t> out(cap);
    b200z_frame_io io{0, src.size(), 0, cap};
    b200z_compress_result res{};
    if (int e = b200z_compress_frames_batch(c, src.data(), src.size(), B200Z_MEM_HOST, &io, 1, level, flags, out.data(), cap, B200Z_MEM_HOST, &res)) return e;
    if (res.status) return res.status;
    for (size_t done = 0; done < res.out_size;) {   // write_all
        const long w = wr(wuser, out.data() + done, (size_t)(res.out_size - done));
        if (w <= 0) { c->err = "write callback failed"; return B200Z_ERR_INVALID_ARGUMENT; }
        done += (size_t)w;
    }
    return 0;
}
