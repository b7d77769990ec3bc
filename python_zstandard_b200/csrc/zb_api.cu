// zb_api.cu -- the C ABI of libzb200.so (include/zb200.h): contexts, memory pools, the host
// orchestration that replaces decompress_from_framesources (c-ext/decompressor.c:1186-1455).
//
// The reference partitions the batch over a pthread pool (POOL_add, c-ext/decompressor.c:1290-1320);
// here the partition is the CUDA grid and the "workers" are warps.  What stays on the host is only
// what the reference also does on its calling thread: argument marshalling, output ownership and
// first-error selection.
#include "zb_common.cuh"
#include "../../include/zb200.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <chrono>
#include <cstdlib>
#include <string>
#include <vector>
#include <thread>
#include <map>
#include <algorithm>

extern "C" {
void zb_launch_default_tables(cudaStream_t st);
void zb_launch_scan(const u8* src, const ZbSegment* segs, u32 n, ZbFrameInfo* info, u64 window_limit, u32* big_list, cudaStream_t st);
void zb_launch_scan_blocks(const u8* src, const ZbSegment* segs, u32 n, const ZbFramePlace* place, ZbDictDev dict, u32* status,
                           void* bdesc, u64* frame_end, const u32* big_list, cudaStream_t st);
void zb_launch_entropy_blocks(const u8* src, const void* bdesc, u32 n_blocks, ZbBlock* blocks, ZbSeq* seqs, u8* lits, u32 n_ctas, u32* work_counter,
                              ZbDictDev dict, u32* status, void* bexit, u32 take, cudaStream_t st);
void zb_launch_resolve_blocks(const u8* src, const ZbSegment* segs, u32 n, const ZbFramePlace* place, const ZbFrameInfo* info, const u64* dst_sizes,
                              ZbBlock* blocks, const void* bdesc, const void* bexit, const u64* frame_end, u64 n_blocks, ZbSeq* seqs, ZbDictDev dict,
                              u32* status, u64* out_sizes, u32* ck_expect, u32* entry_rep, cudaStream_t st);
size_t zb_blkdesc_bytes();
size_t zb_blkexit_bytes();
void zb_launch_place(const ZbFrameInfo* info, const u64* dst_sizes, u32 n, ZbFramePlace* place, u64* totals,
                     u32* status, u64* partial, cudaStream_t st);
void zb_launch_entropy(const u8* src, const ZbSegment* segs, u32 n, const ZbFramePlace* place, const u64* dst_sizes,
                       ZbBlock* blocks, ZbSeq* seqs, u8* lits, u32 n_ctas, u32* work_counter,
                       ZbDictDev dict, u32* status, u64* out_sizes, u32* ck_expect, u32 take, u32 warps, cudaStream_t st);
size_t zb_wave_bytes(u64 n_frames, u64 n_blocks);
size_t zb_chase_bytes(u64 n_total);
int zb_launch_execute_chase(const u8* src, const ZbFramePlace* place, const u32* status, const ZbBlock* blocks, const void* bdesc,
                            const ZbSeq* seqs, const u8* lits, u8* dst, u64 lo, u64 hi, u64 n_total, u64 blk_first, u64 blk_last,
                            void* ptr_mem, u32* d_changed, u32 n_ctas, ZbDictDev dict, cudaStream_t st);
void zb_launch_execute_big(const u8* src, const ZbFramePlace* place, const u32* status, const ZbBlock* blocks, const void* bdesc,
                           const ZbSeq* seqs, const u8* lits, u8* dst, u32 first, u32 end, u64 blk_first, u64 blk_last,
                           u64 n_frames, u64 n_blocks, void* wave_mem, u32 n_ctas, ZbDictDev dict, cudaStream_t st);
void zb_launch_verify(const u8* dst, const ZbFramePlace* place, const u64* out_sizes, const ZbFrameInfo* info, const u32* ck_expect,
                      u32 first, u32 end, u32* status, cudaStream_t st);
void zb_launch_execute(const u8* src, const ZbFramePlace* place, const u32* status, const ZbBlock* blocks,
                       const ZbSeq* seqs, const u8* lits, u8* dst, u32 first, u32 end, ZbDictDev dict, cudaStream_t st);
void zb_launch_finish(const ZbFramePlace* place, const u64* out_sizes, const u32* status, u32 n, ZbSegment* out_segs,
                      u32* first_error, cudaStream_t st);
void zb_launch_digest_dict(const u8* dict, u32 n, ZbDictDigest* out, cudaStream_t st);
size_t zb_encode_scratch_bytes();
void zb_launch_compress_blocks(const u8* src, const void* jobs, u32 n_jobs, void* scratch, u32 n_ctas, u8* slots, u64 slot_bytes,
                               void* outs, u32* work_counter, const u8* dict_tail, u32 dict_D, const u16* dict_table, const void* dict_digest, const void* dict_cct,
                               const unsigned long long* upload_progress, unsigned long long upload_total, u32* upload_status, int dual, int small_blocks, cudaStream_t st);
u32 zb_encode_small_max();
void zb_launch_dict_table(const u8* tail, u32 D, u16* table, cudaStream_t st);
u32 zb_encode_ctable_bytes();
void zb_launch_dict_ctables(const void* digest, void* out3, cudaStream_t st);
void zb_launch_frame_layout(const ZbSegment* segs, const void* seginfo, const void* outs, u32 n_segs, u32 checksum, u32 content_size,
                            u32 dict_id, u32 window_log, u64* sizes, ZbSegment* out_segs, u64* total, cudaStream_t st);
void zb_launch_write_frames(const u8* src, const ZbSegment* segs, const void* seginfo, const void* outs, const u8* slots, u64 slot_bytes,
                            u32 n_segs, u32 checksum, u32 content_size, u32 dict_id, u32 window_log, const ZbSegment* out_segs, u8* dst, cudaStream_t st);
u32 zb_encode_smem_bytes();
u32 zb_encode3_record_max();
u32 zb_encode3_records_per_cta();
void zb_launch_compress_recs(const u8* src, const void* jobs, u32 n_jobs, u32 n_ctas, u8* slots, u64 slot_bytes, void* outs, u32* work_counter,
                             const u8* dict_tail, u32 dict_D, const u16* dict_table, const void* dict_digest, const void* dict_cct,
                             const unsigned long long* upload_progress, unsigned long long upload_total, u32* upload_status, cudaStream_t st);
size_t zb_encode2_scratch_bytes();
void zb_launch_compress_smem(const u8* src, const void* jobs, u32 n_jobs, void* scratch, u32 n_ctas, u8* slots, u64 slot_bytes, void* outs, u32* work_counter,
                             const unsigned long long* upload_progress, unsigned long long upload_total, u32* upload_status, cudaStream_t st);
}

namespace {

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;          // grow-only with slack
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return (T*)p; }
};

struct PinnedBlock { void* p; size_t cap; bool busy; };

}  // namespace

struct zb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;          // device->host copies of finished chunks, overlapping later chunks' kernels
    cudaEvent_t chunk_ev[64] = {nullptr};
    unsigned long long* h_progress = nullptr;    // pinned: the byte counts the chunked upload publishes to the compress kernel
    std::string last_error;
    int sm_count = 148;
    // device arenas (grow-only)
    DevBuf src, segs, dst_sizes, info, place, status, out_sizes, blocks, seqs, lits, dst, lane, small, out_segs, partial;
    DevBuf jobs, seginfo, slots, bouts, escratch, fsizes, ck;
    DevBuf bdesc, bexit, erep, fend, wave;    // block-parallel decode path
    DevBuf biglist;                           // frames whose scans are a warp's work (zb_scan_frames_big)
    DevBuf chase;                             // its pointer-jumping execute stage: a source pointer per output byte
    int last_chase_rounds = 0;
    const char* last_compress_kernel = "";    // which of the three block kernels the last compress call ran (profile slot zb_compress_blocks)
    u32 entropy_warps = 0;
    // pinned pool
    std::mutex mu;
    std::vector<PinnedBlock> pinned;
    // profiling
    bool prof = false;
    std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0;
    struct Span { int k; cudaEvent_t a, b; };
    std::vector<Span> spans;
    float k_ms[ZB200_K_COUNT] = {0}; u32 k_launch[ZB200_K_COUNT] = {0};
    u64 last_scratch = 0;
    int live_results = 0;
};

struct zb200_ddict {
    zb200_ctx* ctx; void* d_raw = nullptr; ZbDictDigest* d_digest = nullptr; ZbDictDev dev; size_t size = 0;
    u16* d_ctable = nullptr; const u8* c_tail = nullptr; u32 c_D = 0; void* d_cct = nullptr;      // compression view: last <= 32 KiB of the content + its hash table
};

struct zb200_result {
    zb200_ctx* ctx; void* data = nullptr; bool data_on_device = false; bool data_pinned_pool = false;
    bool data_owned_device = false;        // ZB200_DST_DEVICE: the result owns its device allocation (stream-ordered pool)
    u64 size = 0; size_t n = 0;
    std::vector<zb200_segment> segs;
    bool has_error = false; size_t err_item = 0; int err_code = 0; u64 err_got = 0, err_expected = 0;
};

namespace {

int fail(zb200_ctx* c, const char* what, cudaError_t e)
{
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s", what, e == cudaSuccess ? "invalid argument" : cudaGetErrorString(e));
    if (c) c->last_error = buf;
    return -1;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, #call, e_); } while (0)

cudaEvent_t get_event(zb200_ctx* c)
{
    if (c->ev_used == c->ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); c->ev_pool.push_back(e); }
    return c->ev_pool[c->ev_used++];
}
struct KSpan {
    zb200_ctx* c; int k; cudaEvent_t a = nullptr;
    KSpan(zb200_ctx* c_, int k_) : c(c_), k(k_) { if (c->prof) { a = get_event(c); cudaEventRecord(a, c->stream); } c->k_launch[k]++; }
    ~KSpan() { if (c->prof) { cudaEvent_t b = get_event(c); cudaEventRecord(b, c->stream); c->spans.push_back({k, a, b}); } }
};
void fold_spans(zb200_ctx* c)
{
    for (auto& s : c->spans) { float ms = 0; if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) c->k_ms[s.k] += ms; }
    c->spans.clear(); c->ev_used = 0;
}

void* pinned_get(zb200_ctx* c, size_t bytes)
{
    // size classes (powers of two up to 64 MiB, then multiples of 64 MiB) so that batches of slightly different
    // sizes reuse the same blocks; blocks are kept for the life of the context (page-locking is slow)
    size_t cls = 1 << 16;
    while (cls < bytes && cls < ((size_t)64 << 20)) cls <<= 1;
    if (cls < bytes) cls = (bytes + ((size_t)64 << 20) - 1) & ~(((size_t)64 << 20) - 1);
    std::lock_guard<std::mutex> g(c->mu);
    PinnedBlock* best = nullptr;
    for (auto& b : c->pinned) if (!b.busy && b.cap >= cls && (!best || b.cap < best->cap)) best = &b;
    if (best) { best->busy = true; return best->p; }
    void* p = nullptr;
    if (cudaHostAlloc(&p, cls, cudaHostAllocPortable) != cudaSuccess) {
        // out of pinned memory: release idle blocks and retry once
        for (size_t i = 0; i < c->pinned.size();) {
            if (!c->pinned[i].busy) { cudaFreeHost(c->pinned[i].p); c->pinned.erase(c->pinned.begin() + (long)i); } else i++;
        }
        if (cudaHostAlloc(&p, cls, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    }
    c->pinned.push_back({p, cls, true});
    return p;
}
void pinned_put(zb200_ctx* c, void* p)
{
    std::lock_guard<std::mutex> g(c->mu);
    for (auto& b : c->pinned) if (b.p == p) { b.busy = false; return; }
}
bool zb_trace_on() { static int v = -1; if (v < 0) { const char* e = getenv("ZB200_TRACE"); v = (e && *e && *e != '0') ? 1 : 0; } return v == 1; }
double zb_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

ZbDictDev no_dict() { ZbDictDev d; memset(&d, 0, sizeof d); return d; }

// One upload at a time per device: when several contexts work on sub-batches of one call, this staggers
// them (A computes and downloads while B uploads) instead of letting them share every stage in lock-step.
std::mutex g_upload_mu[16];

}  // namespace

extern "C" {

int zb200_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

int zb200_ctx_create(int device, zb200_ctx** out)
{
    *out = nullptr;
    int n = zb200_device_count();
    if (n <= 0 || device < 0 || device >= n) return -2;          // no CUDA device: there is no CPU path
    zb200_ctx* ctx = new zb200_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx; return -1;
    }
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    {   // device-resident results come from the stream-ordered pool: keep what it has freed (no cudaMalloc per call)
        cudaMemPool_t pool; unsigned long long keep = ~0ull;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (auto& e : ctx->chunk_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaHostAlloc((void**)&ctx->h_progress, 64 * sizeof(unsigned long long), cudaHostAllocPortable);
    zb_launch_default_tables(ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return -1; }
    *out = ctx;
    return 0;
}

void zb200_ctx_destroy(zb200_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->bdesc.release(); ctx->bexit.release(); ctx->erep.release(); ctx->fend.release(); ctx->wave.release(); ctx->chase.release(); ctx->biglist.release();
    DevBuf* all[] = {&ctx->src, &ctx->segs, &ctx->dst_sizes, &ctx->info, &ctx->place, &ctx->status, &ctx->out_sizes,
                     &ctx->blocks, &ctx->seqs, &ctx->lits, &ctx->dst, &ctx->lane, &ctx->small, &ctx->out_segs, &ctx->partial,
                     &ctx->jobs, &ctx->seginfo, &ctx->slots, &ctx->bouts, &ctx->escratch, &ctx->fsizes, &ctx->ck};
    for (auto* b : all) b->release();
    for (auto& b : ctx->pinned) cudaFreeHost(b.p);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    for (auto e : ctx->chunk_ev) if (e) cudaEventDestroy(e);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->h_progress) cudaFreeHost(ctx->h_progress);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* zb200_ctx_last_error(const zb200_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "no context"; }
void* zb200_ctx_stream(zb200_ctx* ctx) { return (void*)ctx->stream; }
int zb200_ctx_synchronize(zb200_ctx* ctx) { cudaSetDevice(ctx->device); CK(cudaStreamSynchronize(ctx->stream)); return 0; }

const char* zb200_error_string(int code)
{
    // strings of ERR_getErrorString (zstd/zstd.c, error_private.c) so messages match the reference's
    switch (code) {
    case 0: return "No error detected";
    case 1: return "Error (generic)";
    case 10: return "Unknown frame descriptor";
    case 12: return "Version not supported";
    case 14: return "Unsupported frame parameter";
    case 16: return "Frame requires too much memory for decoding";
    case 20: return "Data corruption detected";
    case 22: return "Restored data doesn't match checksum";
    case 24: return "Header of Literals' block doesn't respect format specification";
    case 30: return "Dictionary is corrupted";
    case 32: return "Dictionary mismatch";
    case 40: return "Unsupported parameter";
    case 42: return "Parameter is out of bound";
    case 44: return "tableLog requires too much memory : unsupported";
    case 46: return "Unsupported max Symbol Value : too large";
    case 48: return "Specified maxSymbolValue is too small";
    case 64: return "Allocation error : not enough memory";      /* also: a frame whose literal / sequence counts do not fit 32 bits */
    case 70: return "Destination buffer is too small";
    case 72: return "Src size is incorrect";
    case 74: return "Operation on NULL destination buffer";
    case ZB200_E_UNKNOWN_SIZE: return "could not determine decompressed size";
    case ZB200_E_SIZE_MISMATCH: return "decompressed size mismatch";
    default: return "Unspecified error code";
    }
}

void* zb200_host_alloc(zb200_ctx* ctx, size_t bytes) { cudaSetDevice(ctx->device); return pinned_get(ctx, bytes ? bytes : 1); }
void  zb200_host_free(zb200_ctx* ctx, void* p) { pinned_put(ctx, p); }
void* zb200_device_alloc(zb200_ctx* ctx, size_t bytes)
{
    cudaSetDevice(ctx->device); void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void zb200_device_free(zb200_ctx* ctx, void* p) { cudaSetDevice(ctx->device); cudaFree(p); }
int zb200_memcpy_h2d(zb200_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    cudaSetDevice(ctx->device);
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream)); CK(cudaStreamSynchronize(ctx->stream)); return 0;
}
int zb200_memcpy_d2h(zb200_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    cudaSetDevice(ctx->device);
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream)); CK(cudaStreamSynchronize(ctx->stream)); return 0;
}

void zb200_host_copy(void* dst, const void* src, size_t bytes)
{
    size_t const piece = 1u << 20;
    unsigned hw = std::thread::hardware_concurrency(); if (hw == 0) hw = 4;
    size_t nt = bytes / piece; if (nt > 16) nt = 16; if (nt > hw) nt = hw;
    if (nt < 2) { memcpy(dst, src, bytes); return; }
    size_t const n_pieces = (bytes + piece - 1) / piece;
    std::vector<std::thread> th;
    for (size_t t = 0; t < nt; t++)
        th.emplace_back([=] {
            for (size_t k = t; k < n_pieces; k += nt) {
                size_t const o = k * piece, len = o + piece <= bytes ? piece : bytes - o;
                memcpy((char*)dst + o, (const char*)src + o, len);
            }
        });
    for (auto& x : th) x.join();
}

int zb200_pointer_device(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return -1; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged ? a.device : -1;
}

// ---------------------------------------------------------------- dictionaries
int zb200_ddict_create(zb200_ctx* ctx, const void* dict, size_t size, zb200_ddict** out)
{
    *out = nullptr;
    if (!ctx || !dict || size == 0 || size > 0x7FFFFFFFu) return fail(ctx, "zb200_ddict_create", cudaSuccess);
    cudaSetDevice(ctx->device);
    zb200_ddict* d = new zb200_ddict(); d->ctx = ctx; d->size = size;
    cudaError_t e = cudaMalloc(&d->d_raw, size + 16);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d->d_digest, sizeof(ZbDictDigest));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d->d_raw, dict, size, cudaMemcpyHostToDevice, ctx->stream);
    ZbDictDigest* h = nullptr;
    if (e == cudaSuccess) {
        zb_launch_digest_dict((const u8*)d->d_raw, (u32)size, d->d_digest, ctx->stream);
        h = (ZbDictDigest*)malloc(sizeof(ZbDictDigest));
        e = cudaMemcpyAsync(h, d->d_digest, sizeof(ZbDictDigest), cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { free(h); zb200_ddict_free(d); return fail(ctx, "zb200_ddict_create", e); }
    if (h->status != ZB_OK) { int code = (int)h->status; free(h); zb200_ddict_free(d); ctx->last_error = zb200_error_string(code); return -code; }
    ZbDictDev& v = d->dev; memset(&v, 0, sizeof v);
    v.content = (const u8*)d->d_raw + h->content_off; v.content_size = (u32)size - h->content_off;
    v.dict_id = h->dict_id; v.has_entropy = h->has_entropy;
    v.huf = d->d_digest->huf; v.huf_log = h->huf_log;
    v.ll = d->d_digest->ll; v.of = d->d_digest->of; v.ml = d->d_digest->ml;
    v.ll_log = h->ll_log; v.of_log = h->of_log; v.ml_log = h->ml_log;
    v.rep[0] = h->rep[0]; v.rep[1] = h->rep[1]; v.rep[2] = h->rep[2];
    free(h);
    // compression view (built now, it is one tiny launch)
    d->c_D = v.content_size < 32768u ? v.content_size : 32768u;
    d->c_tail = v.content + (v.content_size - d->c_D);
    if (d->c_D >= 8 && cudaMalloc((void**)&d->d_ctable, 16384 * sizeof(u16)) == cudaSuccess) {
        zb_launch_dict_table(d->c_tail, d->c_D, d->d_ctable, ctx->stream);
        if (v.has_entropy && cudaMalloc(&d->d_cct, 3 * (size_t)zb_encode_ctable_bytes()) == cudaSuccess)
            zb_launch_dict_ctables(d->d_digest, d->d_cct, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    } else d->c_D = 0;
    *out = d;
    return 0;
}
void zb200_ddict_free(zb200_ddict* d)
{
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    if (d->d_raw) cudaFree(d->d_raw);
    if (d->d_digest) cudaFree(d->d_digest);
    if (d->d_ctable) cudaFree(d->d_ctable);
    if (d->d_cct) cudaFree(d->d_cct);
    delete d;
}
uint32_t zb200_ddict_id(const zb200_ddict* d) { return d ? d->dev.dict_id : 0; }

// ---------------------------------------------------------------- batch decompression
// Device-side pipeline shared by the host and device entry points.  d_src/d_segs/d_dst_sizes are device
// pointers.  On return the output is in ctx->dst (or caller_dst), segment table + status on the host.
static int run_decompress(zb200_ctx* ctx, const u8* d_src, const ZbSegment* d_segs, size_t n, const u64* d_dst_sizes,
                          const zb200_ddict* dict, zb200_result* res, bool copy_back, bool exact_sizes, u64 window_limit)
{
    u32 const nf = (u32)n;
    ZbDictDev dd = dict ? dict->dev : no_dict();
    CK(ctx->info.ensure(n * sizeof(ZbFrameInfo)));
    CK(ctx->place.ensure((n + 1) * sizeof(ZbFramePlace)));
    CK(ctx->status.ensure(n * sizeof(u32)));
    CK(ctx->out_sizes.ensure(n * sizeof(u64)));
    CK(ctx->out_segs.ensure(n * sizeof(ZbSegment)));
    CK(ctx->small.ensure(512));
    CK(ctx->partial.ensure(((n + 1023) / 1024 + 1) * 4 * sizeof(u64)));
    u64* d_totals = ctx->small.as<u64>();                 // [0..3] totals
    u32* d_counter = (u32*)(d_totals + 8);                // work counter
    u32* d_first_err = d_counter + 1;
    u32 init[2] = {0, 0xFFFFFFFFu};
    CK(cudaMemcpyAsync(d_counter, init, sizeof init, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_totals, 0, 8 * sizeof(u64), ctx->stream));
    CK(ctx->ck.ensure(n * sizeof(u32)));

    CK(ctx->biglist.ensure(((size_t)n + 1) * sizeof(u32)));
    { KSpan s(ctx, ZB200_K_SCAN); zb_launch_scan(d_src, d_segs, nf, ctx->info.as<ZbFrameInfo>(), window_limit, ctx->biglist.as<u32>(), ctx->stream); }
    { KSpan s(ctx, ZB200_K_PLACE);
      zb_launch_place(ctx->info.as<ZbFrameInfo>(), d_dst_sizes, nf, ctx->place.as<ZbFramePlace>(), d_totals,
                      ctx->status.as<u32>(), ctx->partial.as<u64>(), ctx->stream); }
    u64 totals[5];
    CK(cudaMemcpyAsync(totals, d_totals, sizeof totals, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));

    // persistent entropy grid: one CTA per SM (its shared memory holds the decode tables); trimmed per chunk below
    u32 const ctas = (u32)ctx->sm_count;
    CK(ctx->blocks.ensure((totals[1] + 1) * sizeof(ZbBlock)));
    CK(ctx->seqs.ensure((totals[2] + 1) * sizeof(ZbSeq)));
    CK(ctx->lits.ensure(totals[3] + 64));
    // the output: the context's arena when it is copied back to the host, an allocation of its own (stream-ordered pool)
    // when the caller keeps it on the device -- the next call on this context must not touch a live result
    u8* d_out;
    if (copy_back) { CK(ctx->dst.ensure(totals[0] + 64)); d_out = ctx->dst.as<u8>(); }
    else { void* p = nullptr; CK(cudaMallocAsync(&p, totals[0] + 64, ctx->stream)); d_out = (u8*)p; res->data = p; res->data_on_device = true; res->data_owned_device = true; }
    ctx->last_scratch = (totals[1] + 1) * sizeof(ZbBlock) + (totals[2] + 1) * sizeof(ZbSeq) + totals[3];

    // ---- chunks of frames: the device->host copy of chunk k overlaps the kernels of chunk k+1
    u32 n_chunks = 1;
    if (copy_back) { u64 c = totals[0] / (48ull << 20); n_chunks = (u32)(c < 1 ? 1 : (c > 32 ? 32 : c)); if (n_chunks > nf) n_chunks = nf; }
    std::vector<u32> cut(n_chunks + 1); for (u32 k = 0; k <= n_chunks; k++) cut[k] = (u32)((u64)nf * k / n_chunks);
    std::vector<ZbFramePlace> cpl(n_chunks + 1);
    if (n_chunks > 1) {
        for (u32 k = 0; k <= n_chunks; k++)
            CK(cudaMemcpyAsync(&cpl[k], ctx->place.as<ZbFramePlace>() + cut[k], sizeof(ZbFramePlace), cudaMemcpyDeviceToHost, ctx->stream));
        std::vector<u32> cinit(n_chunks); for (u32 k = 0; k < n_chunks; k++) cinit[k] = cut[k];
        CK(cudaMemcpyAsync(d_counter + 8, cinit.data(), n_chunks * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    // Frames of several blocks when the batch alone does not fill the machine (one huge frame at the limit): a lane per BLOCK
    // instead of a lane per frame for the entropy stage (zb_scan_blocks -> zb_entropy_blocks -> zb_resolve_blocks / zb_patch_blocks)
    // Measured (tools/gpu_c3_decode.py, tools/gpu_c5_frame.py): frames of one 128 KiB chunk -- the reference's single block or
    // our ten sub-blocks -- are faster a lane per frame at any batch size (2048 of ours: 18.4 vs 6.6 GB/s); from a few full
    // blocks per frame on the lane's serial chain (4-5 ms per 128 KiB) is what the block path removes.
    int const force_blocks = getenv("ZB200_BLOCK_PATH") ? atoi(getenv("ZB200_BLOCK_PATH")) : -1;      // (read per call: tests switch it)
    bool const block_path = force_blocks >= 0 ? force_blocks != 0 : (totals[1] > n && n < 3000 && totals[0] >= (u64)n * (512u << 10));
    bool chase_path = false;
    ctx->last_chase_rounds = 0;
    if (block_path) {
        u64 const nb = totals[1];
        CK(ctx->bdesc.ensure((nb + 1) * zb_blkdesc_bytes()));
        CK(ctx->bexit.ensure((nb + 1) * zb_blkexit_bytes()));
        CK(ctx->erep.ensure((nb + 1) * 3 * sizeof(u32)));
        CK(ctx->fend.ensure(n * sizeof(u64)));
        CK(ctx->wave.ensure(zb_wave_bytes(nf, nb)));
        // FEW frames of many blocks (one huge frame at the limit): the copy-execute chain of a frame is serial however it is
        // mapped, so it is shortened by pointer doubling instead (zb_chase_*); many frames keep the machine busy frame-parallel
        int const force_chase = getenv("ZB200_CHASE") ? atoi(getenv("ZB200_CHASE")) : -1;
        chase_path = force_chase >= 0 ? force_chase != 0 : (nf < 64 && nb >= 8ull * nf);
        if (chase_path && ctx->chase.ensure(zb_chase_bytes(totals[0])) != cudaSuccess) { cudaGetLastError(); chase_path = false; }
        { KSpan s(ctx, ZB200_K_SCAN);
          zb_launch_scan_blocks(d_src, d_segs, nf, ctx->place.as<ZbFramePlace>(), dd, ctx->status.as<u32>(), ctx->bdesc.p, ctx->fend.as<u64>(), ctx->biglist.as<u32>(), ctx->stream); }
        u32 const take = 3, EW = 7;
        u32 cc = ctas; { u64 const need = (nb + EW * take - 1) / (EW * take); if (cc > need) cc = (u32)need; if (cc == 0) cc = 1; }
        { KSpan s(ctx, ZB200_K_ENTROPY);
          zb_launch_entropy_blocks(d_src, ctx->bdesc.p, (u32)nb, ctx->blocks.as<ZbBlock>(), ctx->seqs.as<ZbSeq>(), ctx->lits.as<u8>(), cc, d_counter, dd,
                                   ctx->status.as<u32>(), ctx->bexit.p, take, ctx->stream); }
        { KSpan s(ctx, ZB200_K_PLACE);
          zb_launch_resolve_blocks(d_src, d_segs, nf, ctx->place.as<ZbFramePlace>(), ctx->info.as<ZbFrameInfo>(), exact_sizes ? d_dst_sizes : nullptr,
                                   ctx->blocks.as<ZbBlock>(), ctx->bdesc.p, ctx->bexit.p, ctx->fend.as<u64>(), nb, ctx->seqs.as<ZbSeq>(), dd,
                                   ctx->status.as<u32>(), ctx->out_sizes.as<u64>(), ctx->ck.as<u32>(), ctx->erep.as<u32>(), ctx->stream); }
    }
    res->n = n; res->size = totals[0];
    res->segs.resize(n);
    if (copy_back) {
        res->data = pinned_get(ctx, totals[0] ? totals[0] : 1);
        if (!res->data) return fail(ctx, "pinned output allocation", cudaErrorMemoryAllocation);
        res->data_pinned_pool = true;
    }
    for (u32 k = 0; k < n_chunks; k++) {
        u32 const f0 = cut[k], f1 = cut[k + 1];
        u32* const counter = n_chunks > 1 ? d_counter + 8 + k : d_counter;
        // frames per warp: large frames carry large decode tables (a 128 KiB block: ~4 KB Huffman + ~5 KB FSE cells per lane)
        u64 const avg_out = (cpl.size() > 1 && n_chunks > 1 ? (cpl[k + 1].dst_off - cpl[k].dst_off) : totals[0]) / (f1 - f0 ? f1 - f0 : 1);
        u32 const EW = avg_out <= (8u << 10) ? 8u : 7u;          // warps per CTA: see zb_entropy.cuh
        u32 take = avg_out <= (8u << 10) ? 32u : (avg_out <= (16u << 10) ? 16u : (avg_out <= (32u << 10) ? 8u : (avg_out <= (64u << 10) ? 4u : 3u)));
        // small batches: spread the frames over all resident warps rather than filling few warps' lanes
        { u32 const spread = (f1 - f0 + ctas * EW - 1) / (ctas * EW); if (take > spread) take = spread ? spread : 1; }
        u32 cc = ctas; { u32 const need = (f1 - f0 + EW * take - 1) / (EW * take); if (cc > need) cc = need; if (cc == 0) cc = 1; }
        if (!block_path) { KSpan s(ctx, ZB200_K_ENTROPY);
          zb_launch_entropy(d_src, d_segs, f1, ctx->place.as<ZbFramePlace>(), exact_sizes ? d_dst_sizes : nullptr, ctx->blocks.as<ZbBlock>(),
                            ctx->seqs.as<ZbSeq>(), ctx->lits.as<u8>(), cc, counter, dd,
                            ctx->status.as<u32>(), ctx->out_sizes.as<u64>(), ctx->ck.as<u32>(), take, EW, ctx->stream); }
        { KSpan s(ctx, ZB200_K_EXECUTE);
          if (chase_path) {
              int const r = zb_launch_execute_chase(d_src, ctx->place.as<ZbFramePlace>(), ctx->status.as<u32>(), ctx->blocks.as<ZbBlock>(), ctx->bdesc.p,
                                                    ctx->seqs.as<ZbSeq>(), ctx->lits.as<u8>(), d_out,
                                                    n_chunks > 1 ? cpl[k].dst_off : 0, n_chunks > 1 ? cpl[k + 1].dst_off : totals[0], totals[0],
                                                    n_chunks > 1 ? cpl[k].blk_off : 0, n_chunks > 1 ? cpl[k + 1].blk_off : totals[1],
                                                    ctx->chase.p, d_counter + 48, ctas, dd, ctx->stream);
              if (r < 0) return fail(ctx, "pointer-jumping execute", cudaGetLastError());
              ctx->last_chase_rounds = r;
          }
          else if (block_path) zb_launch_execute_big(d_src, ctx->place.as<ZbFramePlace>(), ctx->status.as<u32>(), ctx->blocks.as<ZbBlock>(), ctx->bdesc.p,
                                                ctx->seqs.as<ZbSeq>(), ctx->lits.as<u8>(), d_out, f0, f1,
                                                n_chunks > 1 ? cpl[k].blk_off : 0, n_chunks > 1 ? cpl[k + 1].blk_off : totals[1],
                                                nf, totals[1], ctx->wave.p, ctas, dd, ctx->stream);
          else zb_launch_execute(d_src, ctx->place.as<ZbFramePlace>(), ctx->status.as<u32>(), ctx->blocks.as<ZbBlock>(),
                                 ctx->seqs.as<ZbSeq>(), ctx->lits.as<u8>(), d_out, f0, f1, dd, ctx->stream); }
        if (totals[4]) { KSpan s(ctx, ZB200_K_VERIFY);
          zb_launch_verify(d_out, ctx->place.as<ZbFramePlace>(), ctx->out_sizes.as<u64>(), ctx->info.as<ZbFrameInfo>(),
                           ctx->ck.as<u32>(), f0, f1, ctx->status.as<u32>(), ctx->stream); }
        if (copy_back && n_chunks > 1) {
            CK(cudaEventRecord(ctx->chunk_ev[k], ctx->stream));
            CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->chunk_ev[k], 0));
            u64 const o0 = cpl[k].dst_off, o1 = cpl[k + 1].dst_off;
            if (o1 > o0) CK(cudaMemcpyAsync((u8*)res->data + o0, d_out + o0, o1 - o0, cudaMemcpyDeviceToHost, ctx->copy_stream));
        }
    }
    { KSpan s(ctx, ZB200_K_FINISH);
      zb_launch_finish(ctx->place.as<ZbFramePlace>(), ctx->out_sizes.as<u64>(), ctx->status.as<u32>(), nf,
                       ctx->out_segs.as<ZbSegment>(), d_first_err, ctx->stream); }
    u32 first_err = 0xFFFFFFFFu;
    CK(cudaMemcpyAsync(res->segs.data(), ctx->out_segs.p, n * sizeof(ZbSegment), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&first_err, d_first_err, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    if (copy_back && n_chunks == 1) CK(cudaMemcpyAsync(res->data, d_out, totals[0], cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (copy_back && n_chunks > 1) CK(cudaStreamSynchronize(ctx->copy_stream));
    if (ctx->prof) fold_spans(ctx);
    if (first_err != 0xFFFFFFFFu) {
        u32 code = 0; u64 got = 0; ZbFramePlace pl;
        cudaMemcpy(&code, ctx->status.as<u32>() + first_err, sizeof code, cudaMemcpyDeviceToHost);
        cudaMemcpy(&pl, ctx->place.as<ZbFramePlace>() + first_err, sizeof pl, cudaMemcpyDeviceToHost);
        cudaMemcpy(&got, ctx->out_sizes.as<u64>() + first_err, sizeof got, cudaMemcpyDeviceToHost);     // what the frame regenerated (size mismatch)
        res->has_error = true; res->err_item = first_err; res->err_code = (int)code; res->err_got = got; res->err_expected = pl.dst_cap;
    }
    return 0;
}

static u64 window_limit_of(const zb200_dparams* p)
{
    // ZSTD_MAXWINDOWSIZE_DEFAULT = (1 << ZSTD_WINDOWLOG_LIMIT_DEFAULT) + 1 (zstd/zstd.c:43465, :5585)
    return p && p->max_window_size ? p->max_window_size : ((1ull << 27) + 1);
}

static int decompress_common(zb200_ctx* ctx, const void* src_base, const zb200_segment* segs, size_t n,
                             const uint64_t* dst_sizes, const zb200_ddict* dict, uint32_t flags, zb200_result** out,
                             const zb200_dparams* dparams = nullptr)
{
    *out = nullptr;
    if (!ctx || !segs || n == 0 || n > 0x7FFFFFF0u) return fail(ctx, "zb200_decompress_batch: bad arguments", cudaSuccess);
    cudaSetDevice(ctx->device);
    const u8* d_src; const ZbSegment* d_segs; const u64* d_dst_sizes = nullptr;
    if ((flags & ZB200_SRC_DEVICE) && (flags & ZB200_SEGS_HOST)) {
        // the frames are on the device, their table (and the sizes) on the host: only those are uploaded
        CK(ctx->segs.ensure(n * sizeof(ZbSegment)));
        if (dst_sizes) CK(ctx->dst_sizes.ensure(n * sizeof(u64)));
        CK(cudaMemcpyAsync(ctx->segs.p, segs, n * sizeof(ZbSegment), cudaMemcpyHostToDevice, ctx->stream));
        if (dst_sizes) CK(cudaMemcpyAsync(ctx->dst_sizes.p, dst_sizes, n * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));          // (the caller's tables may go away)
        d_src = (const u8*)src_base; d_segs = ctx->segs.as<ZbSegment>();
        if (dst_sizes) d_dst_sizes = ctx->dst_sizes.as<u64>();
    } else if (flags & ZB200_SRC_DEVICE) {
        d_src = (const u8*)src_base; d_segs = (const ZbSegment*)segs; d_dst_sizes = dst_sizes;
    } else {
        // host input: one contiguous copy of the referenced span (the data a BufferWithSegments holds)
        u64 lo = ~0ull, hi = 0;
        for (size_t i = 0; i < n; i++) { if (segs[i].offset < lo) lo = segs[i].offset; if (segs[i].offset + segs[i].length > hi) hi = segs[i].offset + segs[i].length; }
        if (hi < lo) { lo = hi = 0; }
        CK(ctx->src.ensure(hi - lo + 64));
        CK(ctx->segs.ensure(n * sizeof(ZbSegment)));
        if (dst_sizes) CK(ctx->dst_sizes.ensure(n * sizeof(u64)));
        std::vector<zb200_segment> tmp;
        {
            std::lock_guard<std::mutex> up(g_upload_mu[ctx->device & 15]);
            CK(cudaMemcpyAsync(ctx->src.p, (const u8*)src_base + lo, hi - lo, cudaMemcpyHostToDevice, ctx->stream));
            if (lo == 0) CK(cudaMemcpyAsync(ctx->segs.p, segs, n * sizeof(ZbSegment), cudaMemcpyHostToDevice, ctx->stream));
            else {
                tmp.assign(segs, segs + n);
                for (auto& s : tmp) s.offset -= lo;
                CK(cudaMemcpyAsync(ctx->segs.p, tmp.data(), n * sizeof(ZbSegment), cudaMemcpyHostToDevice, ctx->stream));
            }
            if (dst_sizes) CK(cudaMemcpyAsync(ctx->dst_sizes.p, dst_sizes, n * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
        d_src = ctx->src.as<u8>(); d_segs = ctx->segs.as<ZbSegment>();
        if (dst_sizes) d_dst_sizes = ctx->dst_sizes.as<u64>();
    }
    zb200_result* res = new zb200_result(); res->ctx = ctx;
    int rc = run_decompress(ctx, d_src, d_segs, n, d_dst_sizes, dict, res, !(flags & ZB200_DST_DEVICE),
                            !(flags & ZB200_SIZES_ARE_CAPACITY), window_limit_of(dparams));
    if (rc) { zb200_result_free(res); return rc; }
    *out = res;
    return 0;
}

int zb200_decompress_batch(zb200_ctx* ctx, const void* src_base, const zb200_segment* segs, size_t n,
                           const uint64_t* dst_sizes, const zb200_ddict* dict, uint32_t flags, zb200_result** out)
{
    return decompress_common(ctx, src_base, segs, n, dst_sizes, dict, flags, out);
}

int zb200_decompress_batch_ex(zb200_ctx* ctx, const void* src_base, const zb200_segment* segs, size_t n,
                              const uint64_t* dst_sizes, const zb200_ddict* dict, const zb200_dparams* params, uint32_t flags, zb200_result** out)
{
    return decompress_common(ctx, src_base, segs, n, dst_sizes, dict, flags, out, params);
}

int zb200_decompress_batch_ptrs(zb200_ctx* ctx, const void* const* srcs, const size_t* sizes, size_t n,
                                const uint64_t* dst_sizes, const zb200_ddict* dict, uint32_t flags, zb200_result** out)
{
    return zb200_decompress_batch_ptrs_ex(ctx, srcs, sizes, n, dst_sizes, dict, nullptr, flags, out);
}

int zb200_decompress_batch_ptrs_ex(zb200_ctx* ctx, const void* const* srcs, const size_t* sizes, size_t n,
                                   const uint64_t* dst_sizes, const zb200_ddict* dict, const zb200_dparams* params, uint32_t flags, zb200_result** out)
{
    *out = nullptr;
    if (!ctx || !srcs || !sizes || n == 0) return fail(ctx, "zb200_decompress_batch_ptrs: bad arguments", cudaSuccess);
    cudaSetDevice(ctx->device);
    // gather the independent buffers into pinned staging (this is the copy a list-of-bytes input costs anyway)
    u64 total = 0; for (size_t i = 0; i < n; i++) total += sizes[i];
    u8* stage = (u8*)pinned_get(ctx, total ? total : 1);
    if (!stage) return fail(ctx, "pinned staging allocation", cudaErrorMemoryAllocation);
    std::vector<zb200_segment> segs(n); u64 pos = 0;
    for (size_t i = 0; i < n; i++) { memcpy(stage + pos, srcs[i], sizes[i]); segs[i].offset = pos; segs[i].length = sizes[i]; pos += sizes[i]; }
    int rc = decompress_common(ctx, stage, segs.data(), n, dst_sizes, dict, flags & ~ZB200_SRC_DEVICE, out, params);
    pinned_put(ctx, stage);
    return rc;
}


// ---------------------------------------------------------------- batch compression
namespace {
struct HostJob { u64 src_pos; u32 size, seg, last, first; };
struct HostSegInfo { u64 first_job; u32 n_jobs, pad; };
}

static int compress_common(zb200_ctx* ctx, const void* src_base, const zb200_segment* segs, size_t n,
                           const zb200_cparams* params, const zb200_ddict* dict, uint32_t flags, zb200_result** out)
{
    *out = nullptr;
    if (!ctx || !segs || n == 0 || n > 0x7FFFFFF0u) return fail(ctx, "zb200_compress_batch: bad arguments", cudaSuccess);
    cudaSetDevice(ctx->device);
    double const tr0 = zb_trace_on() ? zb_now_ms() : 0; double tr1 = 0, tr2 = 0;
    zb200_cparams P; if (params) P = *params; else { memset(&P, 0, sizeof P); P.level = 3; P.write_content_size = 1; }
    if (P.window_log && (P.window_log < 10 || P.window_log > 31)) return fail(ctx, "zb200_compress_batch: window_log out of range [10, 31]", cudaSuccess);
    // Block_Maximum_Size = min(window, 128 KiB) (ZSTD_getBlockSize, zstd/zstd.c:27478): a small window cuts the blocks, and with
    // them the reach of every match (matches never leave their block here)
    u32 const block_max = P.window_log && P.window_log < 17 ? (1u << P.window_log) : ZB_BLOCK_MAX;
    std::vector<zb200_segment> hsegs;
    const u8* d_src; const ZbSegment* d_segs;
    const u8* up_src = nullptr; u64 up_bytes = 0;          // host input to upload while the kernel runs
    if ((flags & ZB200_SRC_DEVICE) && (flags & ZB200_SEGS_HOST)) {
        hsegs.assign(segs, segs + n);
        CK(ctx->segs.ensure(n * sizeof(ZbSegment)));
        CK(cudaMemcpyAsync(ctx->segs.p, segs, n * sizeof(ZbSegment), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));          // (the caller's table may go away)
        d_src = (const u8*)src_base; d_segs = ctx->segs.as<ZbSegment>();
    } else if (flags & ZB200_SRC_DEVICE) {
        hsegs.resize(n);
        CK(cudaMemcpyAsync(hsegs.data(), segs, n * sizeof(ZbSegment), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        d_src = (const u8*)src_base; d_segs = (const ZbSegment*)segs;
    } else {
        hsegs.assign(segs, segs + n);
        u64 lo = ~0ull, hi = 0;
        for (size_t i = 0; i < n; i++) { if (segs[i].offset < lo) lo = segs[i].offset; if (segs[i].offset + segs[i].length > hi) hi = segs[i].offset + segs[i].length; }
        if (hi < lo) { lo = hi = 0; }
        for (auto& s : hsegs) s.offset -= lo;
        CK(ctx->src.ensure(hi - lo + 512));
        CK(ctx->segs.ensure(n * sizeof(ZbSegment)));
        CK(cudaMemcpyAsync(ctx->segs.p, hsegs.data(), n * sizeof(ZbSegment), cudaMemcpyHostToDevice, ctx->stream));
        // the input itself is uploaded in chunks on the copy stream AFTER the block kernel has been launched: the kernel
        // waits per block for the bytes it needs (ZeUpload), so the upload hides behind the compression of earlier blocks
        up_src = (const u8*)src_base + lo; up_bytes = hi - lo;
        d_src = ctx->src.as<u8>(); d_segs = ctx->segs.as<ZbSegment>();
    }
    if (zb_trace_on()) tr1 = zb_now_ms();
    // block jobs: every <=128 KiB slice of every segment (ZSTD_compress_frameChunk's block loop, zstd/zstd.c:27545)
    std::vector<HostJob> jobs; std::vector<HostSegInfo> sinfo(n);
    jobs.reserve(n);
    u32 max_block = 0;
    for (size_t i = 0; i < n; i++) {
        u64 const len = hsegs[i].length; u64 pos = 0;
        sinfo[i].first_job = jobs.size(); sinfo[i].n_jobs = 0; sinfo[i].pad = 0;
        while (pos < len) {
            u32 const sz = (u32)(len - pos < block_max ? len - pos : block_max);
            HostJob j; j.src_pos = hsegs[i].offset + pos; j.size = sz; j.seg = (u32)i; j.first = pos == 0; j.last = pos + sz == len;
            jobs.push_back(j); sinfo[i].n_jobs++; pos += sz;
            if (sz > max_block) max_block = sz;
        }
    }
    size_t const nj = jobs.size();
    u64 const slot_bytes = ((u64)max_block + (max_block >> 7) + 64 + 15) & ~15ull;
    // Blocks of 8 KiB and more (no dictionary, level-3 class) take the round-2 kernel: one CTA per SM with the block resident in
    // shared memory.  Small blocks, dictionaries and the level >= 4 mode stay on the CTA-per-block kernel (6 CTAs per SM).
    static int const force_v1 = getenv("ZB200_ENCODER_V1") ? atoi(getenv("ZB200_ENCODER_V1")) : 0;
    bool const smem_kernel = !dict && P.level < 4 && max_block >= 8192 && !force_v1;
    // Small records with a full dictionary (config 4): a warp per record, 22 records per SM (zb_encode3.cuh).
    bool const recs_kernel = dict && dict->c_D >= 8 && dict->dev.has_entropy && dict->d_cct && P.level < 4 && nj != 0 &&
                             max_block <= zb_encode3_record_max() && !force_v1;
    u32 ctas = smem_kernel ? (u32)ctx->sm_count : (u32)ctx->sm_count * (227u * 1024u / zb_encode_smem_bytes());
    if (recs_kernel) { ctas = (u32)ctx->sm_count; u32 const need = ((u32)nj + zb_encode3_records_per_cta() - 1) / zb_encode3_records_per_cta(); if (ctas > need) ctas = need; }
    if (ctas > nj) ctas = (u32)nj;
    if (ctas == 0) ctas = 1;
    CK(ctx->jobs.ensure((nj + 1) * sizeof(HostJob)));
    CK(ctx->seginfo.ensure(n * sizeof(HostSegInfo)));
    CK(ctx->slots.ensure((nj + 1) * slot_bytes));
    CK(ctx->bouts.ensure((nj + 1) * 8));
    if (!recs_kernel) CK(ctx->escratch.ensure((size_t)ctas * (smem_kernel ? zb_encode2_scratch_bytes() : zb_encode_scratch_bytes())));
    CK(ctx->fsizes.ensure(n * sizeof(u64)));
    CK(ctx->out_segs.ensure(n * sizeof(ZbSegment)));
    CK(ctx->small.ensure(256));
    u64* d_total = ctx->small.as<u64>();
    u32* d_counter = (u32*)(d_total + 8);
    if (nj) CK(cudaMemcpyAsync(ctx->jobs.p, jobs.data(), nj * sizeof(HostJob), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->seginfo.p, sinfo.data(), n * sizeof(HostSegInfo), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_counter, 0, 64, ctx->stream));                       // work counter, upload status, upload progress
    u32* const d_upstatus = d_counter + 1;
    unsigned long long* const d_progress = (unsigned long long*)(d_counter + 4);
    bool const overlap_upload = up_bytes != 0 && nj != 0 && ctx->h_progress != nullptr;
    if (up_bytes && !overlap_upload) CK(cudaMemcpyAsync(ctx->src.p, up_src, up_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (overlap_upload) {
        // The whole upload is queued BEFORE the compress kernel is launched: the kernel spins until the bytes it needs
        // have landed, so once it runs, its progress must not depend on this thread reaching further API calls (another
        // thread's cudaFree on the same device, say, can hold those back until the kernel ends).
        CK(cudaEventRecord(ctx->chunk_ev[0], ctx->stream)); CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->chunk_ev[0], 0));
        // <= 48 chunks of >= 4 MiB; after each chunk the copy engine also writes the new byte count next to the work counter
        u64 chunk = (up_bytes + 47) / 48; if (chunk < ((u64)4 << 20)) chunk = (u64)4 << 20; chunk = (chunk + 255) & ~(u64)255;
        u32 k = 0;
        for (u64 pos = 0; pos < up_bytes; pos += chunk, k++) {
            u64 const len = up_bytes - pos < chunk ? up_bytes - pos : chunk;
            CK(cudaMemcpyAsync((u8*)ctx->src.p + pos, up_src + pos, len, cudaMemcpyHostToDevice, ctx->copy_stream));
            ctx->h_progress[k] = pos + len;
            CK(cudaMemcpyAsync(d_progress, &ctx->h_progress[k], sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->copy_stream));
        }
    }
    ctx->last_compress_kernel = recs_kernel ? "zb_compress_recs" : (smem_kernel ? "zb_compress_smem" : "zb_compress_blocks");
    if (recs_kernel) { KSpan s(ctx, ZB200_K_COMPRESS);
      zb_launch_compress_recs(d_src, ctx->jobs.p, (u32)nj, ctas, ctx->slots.as<u8>(), slot_bytes, ctx->bouts.p, d_counter,
                              dict->c_tail, dict->c_D, dict->d_ctable, (const void*)dict->d_digest, dict->d_cct,
                              overlap_upload ? d_progress : nullptr, up_bytes, d_upstatus, ctx->stream); }
    else if (nj && smem_kernel) { KSpan s(ctx, ZB200_K_COMPRESS);
      zb_launch_compress_smem(d_src, ctx->jobs.p, (u32)nj, ctx->escratch.p, ctas, ctx->slots.as<u8>(), slot_bytes, ctx->bouts.p, d_counter,
                              overlap_upload ? d_progress : nullptr, up_bytes, d_upstatus, ctx->stream); }
    else if (nj) { KSpan s(ctx, ZB200_K_COMPRESS);
      zb_launch_compress_blocks(d_src, ctx->jobs.p, (u32)nj, ctx->escratch.p, ctas, ctx->slots.as<u8>(), slot_bytes, ctx->bouts.p, d_counter,
                                dict ? dict->c_tail : nullptr, dict ? dict->c_D : 0, dict ? dict->d_ctable : nullptr,
                                (dict && dict->c_D && dict->dev.has_entropy) ? (const void*)dict->d_digest : nullptr, dict ? dict->d_cct : nullptr,
                                overlap_upload ? d_progress : nullptr, up_bytes, d_upstatus, P.level >= 4 ? 1 : 0, max_block <= zb_encode_small_max() ? 1 : 0, ctx->stream); }
    if (overlap_upload) {
        // the layout kernels read the input again (raw blocks): they wait for the whole upload, whatever order the segments came in
        CK(cudaEventRecord(ctx->chunk_ev[1], ctx->copy_stream)); CK(cudaStreamWaitEvent(ctx->stream, ctx->chunk_ev[1], 0));
    }
    { KSpan s(ctx, ZB200_K_LAYOUT);
      zb_launch_frame_layout(d_segs, ctx->seginfo.p, ctx->bouts.p, (u32)n, P.write_checksum ? 1 : 0, P.write_content_size ? 1 : 0, P.dict_id, P.window_log,
                             ctx->fsizes.as<u64>(), ctx->out_segs.as<ZbSegment>(), d_total, ctx->stream); }
    u64 total = 0; u32 upstatus = 0;
    CK(cudaMemcpyAsync(&total, d_total, sizeof total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&upstatus, d_upstatus, sizeof upstatus, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (overlap_upload) CK(cudaStreamSynchronize(ctx->copy_stream));
    if (upstatus) return fail(ctx, "zb200_compress_batch: the input upload did not complete", cudaErrorUnknown);
    if (zb_trace_on()) tr2 = zb_now_ms();
    // the result is held by a unique_ptr until it is handed out: every early return below frees it (and its buffers)
    std::unique_ptr<zb200_result, void (*)(zb200_result*)> res(new zb200_result(), zb200_result_free);
    res->ctx = ctx; res->n = n; res->size = total; res->segs.resize(n);
    u8* d_out;
    if (!(flags & ZB200_DST_DEVICE)) { CK(ctx->dst.ensure(total + 64)); d_out = ctx->dst.as<u8>(); }
    else {      // a device-resident result owns its allocation: later calls on this context leave it alone
        void* p = nullptr; CK(cudaMallocAsync(&p, total + 64, ctx->stream));
        d_out = (u8*)p; res->data = p; res->data_on_device = true; res->data_owned_device = true;
    }
    { KSpan s(ctx, ZB200_K_FRAMES);
      zb_launch_write_frames(d_src, d_segs, ctx->seginfo.p, ctx->bouts.p, ctx->slots.as<u8>(), slot_bytes, (u32)n, P.write_checksum ? 1 : 0,
                             P.write_content_size ? 1 : 0, P.dict_id, P.window_log, ctx->out_segs.as<ZbSegment>(), d_out, ctx->stream); }
    CK(cudaMemcpyAsync(res->segs.data(), ctx->out_segs.p, n * sizeof(ZbSegment), cudaMemcpyDeviceToHost, ctx->stream));
    if (!(flags & ZB200_DST_DEVICE)) {
        res->data = pinned_get(ctx, total ? total : 1);
        if (!res->data) return fail(ctx, "pinned output allocation", cudaErrorMemoryAllocation);
        res->data_pinned_pool = true;
        CK(cudaMemcpyAsync(res->data, d_out, total, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->prof) fold_spans(ctx);
    ctx->last_scratch = (recs_kernel ? 0ull : (u64)ctas * (smem_kernel ? zb_encode2_scratch_bytes() : zb_encode_scratch_bytes())) + nj * slot_bytes;
    if (zb_trace_on()) { double const tr3 = zb_now_ms();
        fprintf(stderr, "[zb200] compress ctx %p n=%zu blocks=%zu: start %.3f upload %.2f kernels %.2f frames+download %.2f ms\n",
                (void*)ctx, n, nj, tr0, tr1 - tr0, tr2 - tr1, tr3 - tr2); }
    *out = res.release();
    return 0;
}

int zb200_compress_batch(zb200_ctx* ctx, const void* src_base, const zb200_segment* segs, size_t n,
                         const zb200_cparams* params, const zb200_ddict* dict, uint32_t flags, zb200_result** out)
{
    return compress_common(ctx, src_base, segs, n, params, dict, flags, out);
}

int zb200_compress_batch_ptrs(zb200_ctx* ctx, const void* const* srcs, const size_t* sizes, size_t n,
                              const zb200_cparams* params, const zb200_ddict* dict, uint32_t flags, zb200_result** out)
{
    *out = nullptr;
    if (!ctx || !srcs || !sizes || n == 0) return fail(ctx, "zb200_compress_batch_ptrs: bad arguments", cudaSuccess);
    cudaSetDevice(ctx->device);
    u64 total = 0; for (size_t i = 0; i < n; i++) total += sizes[i];
    u8* stage = (u8*)pinned_get(ctx, total ? total : 1);
    if (!stage) return fail(ctx, "pinned staging allocation", cudaErrorMemoryAllocation);
    std::vector<zb200_segment> segs(n); u64 pos = 0;
    for (size_t i = 0; i < n; i++) { if (sizes[i]) memcpy(stage + pos, srcs[i], sizes[i]); segs[i].offset = pos; segs[i].length = sizes[i]; pos += sizes[i]; }
    int rc = compress_common(ctx, stage, segs.data(), n, params, dict, flags & ~ZB200_SRC_DEVICE, out);
    pinned_put(ctx, stage);
    return rc;
}

uint64_t zb200_compress_bound(uint64_t n) { return n + (n >> 8) + (n < (128u << 10) ? (((128u << 10) - n) >> 11) : 0); }

const void* zb200_result_data(const zb200_result* r) { return r->data; }
uint64_t zb200_result_size(const zb200_result* r) { return r->size; }
size_t zb200_result_count(const zb200_result* r) { return r->n; }
const zb200_segment* zb200_result_segments(const zb200_result* r) { return r->segs.data(); }
int zb200_result_first_error(const zb200_result* r, size_t* item, int* code, uint64_t* got, uint64_t* expected)
{
    if (!r->has_error) return 0;
    if (item) *item = r->err_item; if (code) *code = r->err_code; if (got) *got = r->err_got; if (expected) *expected = r->err_expected;
    return 1;
}
void zb200_result_free(zb200_result* r)
{
    if (!r) return;
    if (r->data && r->data_pinned_pool) pinned_put(r->ctx, r->data);
    if (r->data && r->data_owned_device) { cudaSetDevice(r->ctx->device); cudaFreeAsync(r->data, r->ctx->stream); }
    delete r;
}

// ---------------------------------------------------------------- frame inspection (host, header only)
int zb200_frame_info(const void* vsrc, size_t n, zb200_frame_info_t* o)
{
    // restates ZSTD_getFrameHeader_advanced, zstd/zstd.c:43668-43778 (same rules as zb_parse_header on the device)
    const u8* s = (const u8*)vsrc;
    memset(o, 0, sizeof *o); o->content_size = ~0ull;
    auto rd = [&](size_t p, int k) { u64 v = 0; for (int i = 0; i < k; i++) v |= (u64)s[p + i] << (8 * i); return v; };
    if (n < 5) { o->status = (n >= 4 && rd(0, 4) != ZB_MAGIC && ((u32)rd(0, 4) & 0xFFFFFFF0u) != ZB_MAGIC_SKIP) ? ZB_E_PREFIX_UNKNOWN : ZB_E_SRCSIZE_WRONG; return 0; }
    u32 magic = (u32)rd(0, 4);
    if (magic != ZB_MAGIC) { o->status = ZB_E_PREFIX_UNKNOWN; return 0; }
    u32 fhd = s[4], single = (fhd >> 5) & 1, did = fhd & 3, fcs = fhd >> 6;
    u32 need = 5 + (single ? 0 : 1) + (did == 3 ? 4 : did) + (fcs == 0 ? (single ? 1 : 0) : (1u << fcs));
    if (n < need) { o->status = ZB_E_SRCSIZE_WRONG; return 0; }
    o->header_size = need;
    if (fhd & 8) { o->status = ZB_E_FRAMEPARAM_UNSUPPORTED; return 0; }
    o->has_checksum = (fhd >> 2) & 1;
    size_t pos = 5;
    if (!single) { u32 wl = s[pos++], wlog = (wl >> 3) + 10; if (wlog > 31) { o->status = ZB_E_WINDOW_TOO_LARGE; return 0; }
                   o->window_size = 1ull << wlog; o->window_size += (o->window_size >> 3) * (wl & 7); }
    if (did) { int k = did == 3 ? 4 : (int)did; o->dict_id = (u32)rd(pos, k); pos += (size_t)k; }
    if (fcs == 0) { if (single) o->content_size = s[pos]; }
    else if (fcs == 1) o->content_size = rd(pos, 2) + 256;
    else if (fcs == 2) o->content_size = rd(pos, 4);
    else o->content_size = rd(pos, 8);
    if (single) o->window_size = o->content_size;
    return 0;
}

// ---------------------------------------------------------------- profiling
void zb200_profile_enable(zb200_ctx* ctx, int on) { ctx->prof = on != 0; }
void zb200_profile_reset(zb200_ctx* ctx) { memset(ctx->k_ms, 0, sizeof ctx->k_ms); memset(ctx->k_launch, 0, sizeof ctx->k_launch); }
int zb200_profile_read(zb200_ctx* ctx, float ms[ZB200_K_COUNT], uint32_t launches[ZB200_K_COUNT])
{
    memcpy(ms, ctx->k_ms, sizeof ctx->k_ms); memcpy(launches, ctx->k_launch, sizeof ctx->k_launch); return 0;
}
const char* zb200_kernel_name(int k)
{
    static const char* names[ZB200_K_COUNT] = {"zb_scan_frames", "zb_place_frames", "zb_entropy_decode", "zb_execute", "zb_finish",
                                                "zb_compress_blocks", "zb_frame_layout", "zb_write_frames", "zb_verify_checksums"};
    return (k >= 0 && k < ZB200_K_COUNT && names[k]) ? names[k] : "";
}
// ---------------------------------------------------------------- one batch over several devices
}  // extern "C"
namespace {
struct MultiSlot { zb200_ctx* ctx = nullptr; std::mutex mu; };
std::mutex g_multi_mu;
std::map<std::pair<int, int>, MultiSlot*> g_multi;      // (device, k-th mention of it in a call) -> its context, kept for the process
thread_local std::string g_multi_err;

MultiSlot* multi_slot(int device, int rep)
{
    std::lock_guard<std::mutex> g(g_multi_mu);
    auto& s = g_multi[std::make_pair(device, rep)];
    if (!s) s = new MultiSlot();
    return s;
}

// contiguous, non-empty ranges balanced by input bytes (the rule of python_zstandard_b200/sharding.py::split_ranges, which
// restates the reference's worker partition, c-ext/compressor.c:1183-1200)
std::vector<size_t> multi_cuts(const zb200_segment* segs, size_t n, size_t parts)
{
    std::vector<size_t> cuts{0};
    if (parts > n) parts = n;
    if (parts > 1 && n >= 2) {
        std::vector<u64> cum(n); u64 acc = 0;
        for (size_t i = 0; i < n; i++) { acc += segs[i].length; cum[i] = acc; }
        for (size_t p = 1; p < parts; p++) {
            u64 const target = (u64)((unsigned __int128)acc * p / parts);
            size_t k = (size_t)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin()) + 1;
            if (k < cuts.back() + 1) k = cuts.back() + 1;
            if (k > n - (parts - p)) k = n - (parts - p);
            cuts.push_back(k);
        }
    }
    cuts.push_back(n);
    return cuts;
}

template <class Call>
int multi_run(const int* devices, int n_devices, const zb200_segment* segs, size_t n, const void* dict, size_t dict_size,
              zb200_result** results, size_t* first_item, Call call)
{
    g_multi_err.clear();
    if (!devices || n_devices <= 0 || !segs || n == 0 || !results) { g_multi_err = "bad arguments"; return -3; }
    for (int k = 0; k < n_devices; k++) { results[k] = nullptr; if (first_item) first_item[k] = n; }
    std::vector<size_t> const cuts = multi_cuts(segs, n, (size_t)n_devices);
    size_t const nr = cuts.size() - 1;
    std::vector<int> rc(nr, 0); std::vector<std::string> msg(nr);
    std::vector<std::thread> th;
    std::map<int, int> seen;
    for (size_t k = 0; k < nr; k++) {
        MultiSlot* const slot = multi_slot(devices[k], seen[devices[k]]++);
        size_t const lo = cuts[k], hi = cuts[k + 1];
        if (first_item) first_item[k] = lo;
        th.emplace_back([=, &rc, &msg] {
            std::lock_guard<std::mutex> g(slot->mu);
            if (!slot->ctx && zb200_ctx_create(devices[k], &slot->ctx) != 0) { rc[k] = -2; msg[k] = "cannot create a context on device " + std::to_string(devices[k]); return; }
            zb200_ddict* dd = nullptr;
            if (dict && dict_size && zb200_ddict_create(slot->ctx, dict, dict_size, &dd) != 0) { rc[k] = -1; msg[k] = zb200_ctx_last_error(slot->ctx); return; }
            rc[k] = call(slot->ctx, lo, hi, dd, &results[k]);
            if (rc[k]) msg[k] = zb200_ctx_last_error(slot->ctx);
            if (dd) zb200_ddict_free(dd);
        });
    }
    for (auto& t : th) t.join();
    for (size_t k = 0; k < nr; k++) if (rc[k]) { g_multi_err = "range " + std::to_string(k) + " (device " + std::to_string(devices[k]) + "): " + msg[k]; return rc[k]; }
    return 0;
}
}  // namespace
extern "C" {

const char* zb200_multi_last_error(void) { return g_multi_err.c_str(); }

int zb200_decompress_batch_multi(const int* devices, int n_devices, const void* src_base, const zb200_segment* segs, size_t n,
                                 const uint64_t* dst_sizes, const void* dict, size_t dict_size, const zb200_dparams* params,
                                 uint32_t flags, zb200_result** results, size_t* first_item)
{
    if (flags & (ZB200_SRC_DEVICE | ZB200_DST_DEVICE | ZB200_SEGS_HOST)) { g_multi_err = "host buffers only"; return -3; }
    return multi_run(devices, n_devices, segs, n, dict, dict_size, results, first_item,
                     [=](zb200_ctx* ctx, size_t lo, size_t hi, zb200_ddict* dd, zb200_result** out) {
                         return zb200_decompress_batch_ex(ctx, src_base, segs + lo, hi - lo, dst_sizes ? dst_sizes + lo : nullptr, dd, params, flags, out);
                     });
}

int zb200_compress_batch_multi(const int* devices, int n_devices, const void* src_base, const zb200_segment* segs, size_t n,
                               const zb200_cparams* params, const void* dict, size_t dict_size, uint32_t flags,
                               zb200_result** results, size_t* first_item)
{
    if (flags & (ZB200_SRC_DEVICE | ZB200_DST_DEVICE | ZB200_SEGS_HOST)) { g_multi_err = "host buffers only"; return -3; }
    return multi_run(devices, n_devices, segs, n, dict, dict_size, results, first_item,
                     [=](zb200_ctx* ctx, size_t lo, size_t hi, zb200_ddict* dd, zb200_result** out) {
                         return zb200_compress_batch(ctx, src_base, segs + lo, hi - lo, params, dd, flags, out);
                     });
}

uint64_t zb200_last_scratch_bytes(const zb200_ctx* ctx) { return ctx->last_scratch; }
int zb200_last_chase_rounds(const zb200_ctx* ctx) { return ctx->last_chase_rounds; }
const char* zb200_last_compress_kernel(const zb200_ctx* ctx) { return ctx->last_compress_kernel; }

}  // extern "C"
