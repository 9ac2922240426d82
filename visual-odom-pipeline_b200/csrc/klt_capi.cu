// C ABI of libklt_b200.so (see include/klt_b200.h): context, pyramid planning, kernel launches
// and the host-pointer entry points that stand in for cv2.calcOpticalFlowPyrLK /
// cv2.buildOpticalFlowPyramid as called from reference src/extractor/extractor.py:44,45,65,66.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <thread>
#include <immintrin.h>
#include <functional>
#include <mutex>
#include <new>
#include <vector>

#include "klt_common.cuh"

using namespace klt;

struct klt_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    char name[128] = {0};
    cudaStream_t stream = nullptr;  // for the *_host entry points
    cudaStream_t stream2 = nullptr; // second copy stream of the *_host entry points
    cudaEvent_t ev2 = nullptr;
    // device workspace of the *_host entry points (grown on demand, never shrunk)
    uint8_t* d_ws = nullptr;
    size_t d_ws_bytes = 0;
    // pinned staging for results (and for pageable inputs)
    uint8_t* h_ws = nullptr;
    uint8_t* h_ws_dev = nullptr;   // device-side alias of h_ws
    size_t h_ws_bytes = 0;
    // guards pyr_scratch and bilateral_tabs, which the device-pointer entry points use as well (they take no host_mutex)
    std::mutex cache_mutex;
    // completion counters of the one-launch pyramid build, one array per stream and geometry (klt_pyramid.cu)
    struct PyrScratch { cudaStream_t stream; unsigned* cnt; unsigned* cnt_dev; long long capacity; unsigned gen; long long key[6]; };
    std::vector<PyrScratch> pyr_scratch;
    // weight tables of the bilateral pre-filter on the device, one per parameter set ever used (never freed before destroy)
    struct BilateralTab { int d; double sigma_color, sigma_space; int radius, n_taps; float* d_tab; };
    std::vector<BilateralTab> bilateral_tabs;
    // Pyramid reuse across host calls (the un-edited reference calls calcOpticalFlowPyrLK four times per frame on the same
    // image pair, extractor.py:44,45,65,66): content hashes of the two uploaded images, 3 rotating slots of 4 words
    // (call k writes slot k % 3, compares with slot (k - 1) % 3, zeroes slot (k + 1) % 3), then the skip counter
    unsigned* d_hash = nullptr;
    unsigned long long reuse_call = 0;
    const void* last_imgs[2] = {nullptr, nullptr};        // host addresses of the last call's images: a repeat is likely only
    long long last_pitch[2] = {0, 0};                     // when the caller passes the same arrays again
    long long reuse_key[7] = {0, 0, 0, 0, 0, 0, 0};      // geometry of the last successful call (0: nothing to reuse)
    // the *_host entry points share the workspaces, streams and events above: one call at a time per context
    std::mutex host_mutex;
    // pinned landing zone + helper threads for PAGEABLE host images (see stage_pageable)
    uint8_t* h_in = nullptr;
    size_t h_in_bytes = 0;
    struct Stager;
    Stager* stager = nullptr;
    // pinned landing zone of klt_frame_step_batch's readback (next counts, bad-count flag); step_mutex serialises the calls
    // that use it
    std::mutex step_mutex;
    uint8_t* h_step = nullptr;
    size_t h_step_bytes = 0;
};

namespace {

#define KLT_CUDA(expr)                                   \
    do {                                                 \
        cudaError_t e__ = (expr);                        \
        if (e__ != cudaSuccess) return (klt_status)e__;  \
    } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Makes the context's device current for the duration of an entry point and restores the caller's device afterwards
// (a torch process that calls e.g. calcOpticalFlowPyrLK(device=1) keeps its own current device).
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) {
            err = cudaSetDevice(dev);
            changed = (err == cudaSuccess);
        }
    }
    ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define KLT_DEVICE_GUARD(ctx)                                  \
    DeviceGuard guard__((ctx)->device);                        \
    if (guard__.err != cudaSuccess) return (klt_status)guard__.err

klt_status cuda_status(cudaError_t e) { return e == cudaErrorMemoryAllocation ? KLT_ERR_OUT_OF_MEMORY : (klt_status)e; }

// Replaces a workspace buffer of the *_host entry points (`size` bytes) by one of at least `bytes` (+25 %, rounded up to
// `granule`).  The old buffer is freed once neither of the context's streams can still be using it.
klt_status grow_ws(klt_ctx* ctx, uint8_t*& buf, size_t& size, size_t bytes, size_t granule,
                   cudaError_t (*alloc)(uint8_t**, size_t), cudaError_t (*free_buf)(void*))
{
    if (buf) {
        KLT_CUDA(cudaStreamSynchronize(ctx->stream));
        KLT_CUDA(cudaStreamSynchronize(ctx->stream2));
        free_buf(buf); buf = nullptr; size = 0;
    }
    bytes = align_up(bytes + bytes / 4, granule);
    const cudaError_t e = alloc(&buf, bytes);
    if (e == cudaSuccess) size = bytes;
    return cuda_status(e);
}

// Sizes the device workspace for a *_host call, which is about to overwrite it: the pyramids kept from the last tracking
// call (reuse_key) are forgotten.  A tracking call passes its key and learns in *kept whether they were its own (same key,
// workspace not regrown); it records its key again once it has completed.  Every other call passes nulls.
klt_status claim_device_ws(klt_ctx* ctx, size_t bytes, const long long* key, bool* kept)
{
    const bool grow = bytes > ctx->d_ws_bytes;
    if (key) *kept = !grow && std::memcmp(key, ctx->reuse_key, sizeof(ctx->reuse_key)) == 0;
    ctx->reuse_key[0] = 0;
    if (!grow) return KLT_OK;
    klt_status s = grow_ws(ctx, ctx->d_ws, ctx->d_ws_bytes, bytes, 1 << 20,
                           [](uint8_t** p, size_t n) { return cudaMalloc(p, n); }, cudaFree);
    if (s != KLT_OK) return s;
    // padding columns / rows of the workspace are read (never used) by the 16-byte granule copies: define them once.
    // The memset runs on the legacy stream, which the context's non-blocking streams do not wait for: synchronise, or it
    // could wipe what the current call is about to upload (seen once as a flaky detection result).
    if (cudaMemset(ctx->d_ws, 0, ctx->d_ws_bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) cudaGetLastError();
    return KLT_OK;
}

klt_status ensure_host_ws(klt_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_ws_bytes) return KLT_OK;
    ctx->h_ws_dev = nullptr;
    klt_status s = grow_ws(ctx, ctx->h_ws, ctx->h_ws_bytes, bytes, 1 << 16,
                           [](uint8_t** p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocMapped); }, cudaFreeHost);
    if (s != KLT_OK) return s;
    void* alias = nullptr;
    if (cudaHostGetDevicePointer(&alias, ctx->h_ws, 0) == cudaSuccess) ctx->h_ws_dev = static_cast<uint8_t*>(alias);
    cudaGetLastError();
    return KLT_OK;
}

// pinned landing zone for pageable inputs (see klt_ctx::Stager)
klt_status ensure_host_in(klt_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_in_bytes) return KLT_OK;
    return grow_ws(ctx, ctx->h_in, ctx->h_in_bytes, bytes, 1 << 16,
                   [](uint8_t** p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocDefault); }, cudaFreeHost);
}

// Bytes from the first pixel of a pitched u8 image to its last: what one linear DMA of the image moves.
size_t raw_span(int64_t pitch, int w, int h) { return (size_t)(h - 1) * (size_t)pitch + (size_t)w; }

// Rows (nearly) packed: one linear DMA of the raw span, padding included, beats a pitched 2-D copy (a 2-D copy of e.g.
// 1241-byte rows reaches a fraction of PCIe bandwidth).
bool near_contiguous(size_t raw, int w, int h) { return raw <= 2 * (size_t)w * (size_t)h; }

// upload a u8 image: one contiguous DMA in the caller's pitch when the rows are (nearly) packed, else a 2-D copy
klt_status upload_u8(uint8_t* dst, int64_t* dpitch, const uint8_t* src, int64_t pitch, int w, int h, cudaStream_t st)
{
    const size_t raw = raw_span(pitch, w, h);
    if (near_contiguous(raw, w, h)) {
        KLT_CUDA(cudaMemcpyAsync(dst, src, raw, cudaMemcpyHostToDevice, st));
        *dpitch = pitch;
    } else {
        KLT_CUDA(cudaMemcpy2DAsync(dst, (size_t)w, src, (size_t)pitch, (size_t)w, (size_t)h, cudaMemcpyHostToDevice, st));
        *dpitch = w;
    }
    return KLT_OK;
}

size_t upload_bytes(int64_t pitch, int w, int h)
{
    const size_t raw = raw_span(pitch, w, h);
    return align_up(near_contiguous(raw, w, h) ? raw : (size_t)w * (size_t)h, 256);
}

// KLT_TRACE set: the host entry points synchronise between their phases and print one "[klt trace]" line per call
bool trace_on() { static const bool on = getenv("KLT_TRACE") != nullptr; return on; }
using Clock = std::chrono::steady_clock;
double us(Clock::time_point a, Clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); }

}  // namespace

// Helper threads that copy PAGEABLE host images into the context's pinned landing zone, slice by slice, while the DMA
// engines already move the finished part (the reference hands the drop-in pageable numpy arrays: the output of
// cv2.bilateralFilter, loader.py:86, and `im.copy()`, pipeline.py:103).  cudaMemcpyAsync from pageable memory makes the
// driver do the same staging single-threaded and synchronously (measured: +38 us on a KITTI pair); here the copy of a
// pair is split over the calling thread and kHelpers helpers.  Helpers spin for a short grace period after a job (the
// reference issues its four calls per frame back to back) and then sleep on a condition variable.
struct klt_ctx::Stager {
    static constexpr int kHelpers = 3;
    static constexpr int kParts = kHelpers + 1;
    std::thread threads[kHelpers];
    std::mutex m;
    std::condition_variable cv;
    std::atomic<unsigned> gen{0};
    std::atomic<int> done[2];
    bool stop = false;
    const uint8_t* src[2] = {nullptr, nullptr};
    uint8_t* dst[2] = {nullptr, nullptr};
    size_t bytes[2] = {0, 0};

    static void slice(size_t total, int part, size_t& off, size_t& len)
    {
        const size_t per = ((total + kParts - 1) / kParts + 63) & ~(size_t)63;
        off = std::min(total, per * (size_t)part);
        len = std::min(total - off, per);
    }
    void copy_part(int job, int part)
    {
        size_t off, len;
        slice(bytes[job], part, off, len);
        if (len) std::memcpy(dst[job] + off, src[job] + off, len);
    }
    void worker(int part)
    {
        unsigned seen = 0;
        for (;;) {
            // grace period: poll for ~200 us before sleeping
            bool got = false;
            const auto t0 = std::chrono::steady_clock::now();
            for (int spin = 0;; ++spin) {
                if (gen.load(std::memory_order_acquire) != seen) { got = true; break; }
                _mm_pause();
                if ((spin & 255) == 255 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(200)) break;
            }
            if (!got) {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return stop || gen.load(std::memory_order_acquire) != seen; });
                if (stop) return;
            }
            seen = gen.load(std::memory_order_acquire);
            if (seen == 0xffffffffu) return;
            copy_part(0, part);
            done[0].fetch_add(1, std::memory_order_release);
            copy_part(1, part);
            done[1].fetch_add(1, std::memory_order_release);
        }
    }
    bool start()
    {
        done[0].store(0); done[1].store(0);
        try {
            for (int i = 0; i < kHelpers; ++i) threads[i] = std::thread(&Stager::worker, this, i);
        } catch (...) {
            shutdown();
            return false;
        }
        return true;
    }
    void shutdown()
    {
        { std::lock_guard<std::mutex> lk(m); stop = true; gen.store(0xffffffffu, std::memory_order_release); }
        cv.notify_all();
        for (auto& t : threads) if (t.joinable()) t.join();
    }
    // publish a job of two copies; the caller then runs part kHelpers of each itself and waits with wait_job()
    void post(const uint8_t* s0, uint8_t* d0, size_t b0, const uint8_t* s1, uint8_t* d1, size_t b1)
    {
        src[0] = s0; dst[0] = d0; bytes[0] = b0; src[1] = s1; dst[1] = d1; bytes[1] = b1;
        done[0].store(0, std::memory_order_relaxed); done[1].store(0, std::memory_order_relaxed);
        {
            std::lock_guard<std::mutex> lk(m);
            unsigned g = gen.load(std::memory_order_relaxed) + 1;
            if (g == 0 || g == 0xffffffffu) g = 1;
            gen.store(g, std::memory_order_release);
        }
        cv.notify_all();
    }
    void finish_job(int job)
    {
        copy_part(job, kHelpers);
        while (done[job].load(std::memory_order_acquire) < kHelpers) _mm_pause();
    }
};

namespace {

// Is this host address ordinary (pageable) memory?  cudaPointerGetAttributes costs about a microsecond, and callers pass
// the same few buffers again and again: the answer is remembered per 4 KB page in a small direct-mapped table.  A stale
// entry (the page was freed and came back as the other kind of memory) only costs speed: a pinned buffer gets staged, or
// a pageable one is handed to the driver's own staging.
bool is_pageable(const void* p)
{
    struct Entry { uintptr_t page; bool pageable; };
    thread_local Entry cache[64] = {};
    const uintptr_t page = reinterpret_cast<uintptr_t>(p) >> 12;
    Entry& e = cache[(page ^ (page >> 6)) & 63];
    if (e.page == page && page != 0) return e.pageable;
    cudaPointerAttributes a;
    const cudaError_t err = cudaPointerGetAttributes(&a, p);
    bool pageable = true;
    if (err != cudaSuccess) cudaGetLastError();
    else pageable = (a.type == cudaMemoryTypeUnregistered);
    e.page = page; e.pageable = pageable;
    return pageable;
}

// Posts the copies of two pageable host buffers into the landing zone (src0 to h_in, src1 to h_in + slot) to the helper
// threads, started on first use, and points src0 / src1 at the copies.  Returns the stager, whose two jobs the caller must
// finish before it reads the copies or returns; nullptr (no helper thread could be started): src0 / src1 unchanged.
klt_ctx::Stager* stage_pageable(klt_ctx* ctx, const uint8_t*& src0, size_t bytes0, const uint8_t*& src1, size_t bytes1, size_t slot)
{
    if (!ctx->stager) {
        ctx->stager = new (std::nothrow) klt_ctx::Stager();
        if (ctx->stager && !ctx->stager->start()) { delete ctx->stager; ctx->stager = nullptr; }
    }
    if (ctx->stager) {
        ctx->stager->post(src0, ctx->h_in, bytes0, src1, ctx->h_in + slot, bytes1);
        src0 = ctx->h_in; src1 = ctx->h_in + slot;
    }
    return ctx->stager;
}

// All levels of the item range in ONE launch (pyr_build_fused_kernel); KLT_ERR_UNSUPPORTED: launch level by level.
struct PyrReuse { const unsigned* hash_new; const unsigned* hash_old; unsigned* hash_clear; unsigned long long* skipped; unsigned mask; };

// The pyrDown steps of a layout: step l reads level l (src, w, h, sp, sb) of item first_item and writes level l + 1 (dst, dp, db).
struct PyrSteps {
    const uint8_t* src[KLT_MAX_LEVELS];
    uint8_t* dst[KLT_MAX_LEVELS];
    int w[KLT_MAX_LEVELS], h[KLT_MAX_LEVELS];
    long long sp[KLT_MAX_LEVELS], sb[KLT_MAX_LEVELS], dp[KLT_MAX_LEVELS], db[KLT_MAX_LEVELS];
    PyrSteps(const uint8_t* d_img, const klt_pyr_layout* lay, uint8_t* d_pyr, int first_item)
    {
        for (int l = 0; l < lay->top; ++l) {
            const klt_level& a = lay->level[l];
            const klt_level& b = lay->level[l + 1];
            src[l] = ((l == 0) ? d_img : d_pyr + a.offset) + (int64_t)first_item * a.batch_stride;
            dst[l] = d_pyr + b.offset + (int64_t)first_item * b.batch_stride;
            w[l] = a.w; h[l] = a.h; sp[l] = a.pitch; sb[l] = a.batch_stride; dp[l] = b.pitch; db[l] = b.batch_stride;
        }
    }
};

// Small batches: all levels of the item range in one launch of pyr_build_cluster_kernel; KLT_ERR_UNSUPPORTED: not a small batch.
klt_status pyr_build_cluster(const uint8_t* d_img, const klt_pyr_layout* lay, uint8_t* d_pyr, int first_item, int n_items,
                             cudaStream_t stream, const PyrReuse* reuse)
{
    const PyrSteps S(d_img, lay, d_pyr, first_item);
    PyrCluster P;
    klt_status s = pyr_cluster_plan(P, lay->top, S.src, S.dst, S.w, S.h, S.sp, S.sb, S.dp, S.db, n_items);
    if (s != KLT_OK) return s;
    if (reuse) { P.hash_new = reuse->hash_new; P.hash_old = reuse->hash_old; P.hash_clear = reuse->hash_clear; P.skipped = reuse->skipped; P.reuse_mask = reuse->mask; }
    return pyr_cluster_launch(P, stream);
}

klt_status pyr_build_one_launch(klt_ctx* ctx, const uint8_t* d_img, const klt_pyr_layout* lay, uint8_t* d_pyr, int first_item,
                                int n_items, cudaStream_t stream, const PyrReuse* reuse = nullptr)
{
    const int n_steps = lay->top;
    const PyrSteps S(d_img, lay, d_pyr, first_item);
    PyrFused P;
    long long n_cnt = 0;
    klt_status s = pyr_fused_plan(P, n_steps, S.src, S.dst, S.w, S.h, S.sp, S.sb, S.dp, S.db, n_items, ctx->sm_count, &n_cnt);
    if (s != KLT_OK) return s;
    // A launch that is being recorded into a CUDA graph must not depend on host-side state (the launch number): it takes
    // the device-side form of the kernel, on a counter array of its own (allocated together with the ordinary one, so a
    // build that ran once on this stream before the capture has prepared it).
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
    const bool device_gen = cap != cudaStreamCaptureStatusNone;
    // the counter layout depends on the geometry only (not on which items are built): one array per stream and geometry
    const long long key[6] = {lay->level[0].w, lay->level[0].h, n_steps, n_items, lay->level[0].pitch, P.s[0].rows};
    std::lock_guard<std::mutex> guard(ctx->cache_mutex);
    klt_ctx::PyrScratch* slot = nullptr;
    for (auto& sc : ctx->pyr_scratch)
        if (sc.stream == stream && std::memcmp(sc.key, key, sizeof(key)) == 0) { slot = &sc; break; }
    const size_t words = ((size_t)(n_cnt > 0 ? n_cnt : 0) + 1) / 2 * 2 + 2;   // counters, then (8-byte aligned) the 64-bit CTA count
    if (!slot) {
        if (device_gen) return KLT_ERR_UNSUPPORTED;   // allocation cannot be captured: the caller gets one launch per level
        if (ctx->pyr_scratch.size() >= 64) {          // many geometries on many streams: recycle (rare; costs a sync)
            KLT_CUDA(cudaDeviceSynchronize());
            for (auto& sc : ctx->pyr_scratch) cudaFree(sc.cnt);
            ctx->pyr_scratch.clear();
        }
        klt_ctx::PyrScratch fresh = {stream, nullptr, nullptr, n_cnt, 0u, {key[0], key[1], key[2], key[3], key[4], key[5]}};
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, 2 * words * sizeof(unsigned));
        if (e != cudaSuccess) return cuda_status(e);
        e = cudaMemset(p, 0, 2 * words * sizeof(unsigned));
        if (e == cudaSuccess) e = cudaDeviceSynchronize();   // the memset is not ordered with non-blocking streams
        if (e != cudaSuccess) { cudaFree(p); return (klt_status)e; }
        fresh.cnt = static_cast<unsigned*>(p);
        fresh.cnt_dev = fresh.cnt + words;
        try { ctx->pyr_scratch.push_back(fresh); } catch (const std::bad_alloc&) { cudaFree(p); return KLT_ERR_OUT_OF_MEMORY; }
        slot = &ctx->pyr_scratch.back();
    }
    // counters are monotonic modulo 2^32 and compared by difference: nothing is ever reset
    if (device_gen) {
        P.cnt = slot->cnt_dev;
        P.gen = 0u;
        P.done = reinterpret_cast<unsigned long long*>(slot->cnt_dev + words - 2);
    } else {
        P.cnt = slot->cnt;
        P.gen = ++slot->gen;
        P.done = nullptr;
    }
    if (reuse) { P.hash_new = reuse->hash_new; P.hash_old = reuse->hash_old; P.hash_clear = reuse->hash_clear; P.skipped = reuse->skipped; P.reuse_mask = reuse->mask; }
    s = pyr_fused_launch(P, device_gen, stream);
    if (s != KLT_OK && !device_gen) --slot->gen;
    return s;
}

// Levels 1..top of a validated layout, the context's device current: a small batch in one cluster launch, else one launch
// when pyr_build_one_launch takes the geometry, else one per level.  *reuse_armed: a one-launch build ran with `reuse` (the
// per-level launches ignore it).
klt_status pyr_build(klt_ctx* ctx, const uint8_t* d_img, const klt_pyr_layout* lay, uint8_t* d_pyr, int first_item, int n_items,
                     cudaStream_t stream, const PyrReuse* reuse = nullptr, bool* reuse_armed = nullptr)
{
    if (reuse_armed) *reuse_armed = false;
    if (lay->top >= 1) {
        klt_status s = pyr_build_cluster(d_img, lay, d_pyr, first_item, n_items, stream, reuse);
        if (reuse_armed) *reuse_armed = reuse && s == KLT_OK;
        if (s != KLT_ERR_UNSUPPORTED) return s;
    }
    if (lay->top >= 2) {
        klt_status s = pyr_build_one_launch(ctx, d_img, lay, d_pyr, first_item, n_items, stream, reuse);
        if (reuse_armed) *reuse_armed = reuse && s == KLT_OK;
        if (s != KLT_ERR_UNSUPPORTED) return s;
    }
    for (int l = 0; l < lay->top; ++l) {
        const klt_level& a = lay->level[l];
        const klt_level& b = lay->level[l + 1];
        const uint8_t* src = ((l == 0) ? d_img : d_pyr + a.offset) + (int64_t)first_item * a.batch_stride;
        klt_status s = pyr_down_launch(src, a.w, a.h, a.pitch, a.batch_stride, d_pyr + b.offset + (int64_t)first_item * b.batch_stride,
                                       b.pitch, b.batch_stride, n_items, ctx->sm_count, stream);
        if (s != KLT_OK) return s;
    }
    return KLT_OK;
}

void make_view(const klt_pyr_layout* lay, const uint8_t* img, const uint8_t* pyr, int first_item, int item_stride, PyrView& v)
{
    v.top = lay->top;
    for (int l = 0; l <= lay->top; ++l) {
        const klt_level& s = lay->level[l];
        v.lv[l].data = ((l == 0) ? img : pyr + s.offset) + (int64_t)first_item * s.batch_stride;
        v.lv[l].batch_stride = s.batch_stride * item_stride;
        v.lv[l].pitch = (int)s.pitch;
        v.lv[l].w = s.w;
        v.lv[l].h = s.h;
        v.lv[l].aligned4 = (((uintptr_t)v.lv[l].data | (uintptr_t)s.pitch | (uintptr_t)s.batch_stride) & 3) == 0;
    }
}

klt_status check_layout(const klt_pyr_layout* lay)
{
    if (!lay || lay->top < 0 || lay->top >= KLT_MAX_LEVELS || lay->batch <= 0) return KLT_ERR_INVALID_ARG;
    for (int l = 0; l <= lay->top; ++l) {
        const klt_level& s = lay->level[l];
        if (s.w <= 0 || s.h <= 0 || s.pitch < s.w || s.pitch > 0x7fffffffLL) return KLT_ERR_INVALID_ARG;
        if (lay->batch > 1 && s.batch_stride < s.pitch * (int64_t)(s.h - 1) + s.w) return KLT_ERR_INVALID_ARG;
    }
    return KLT_OK;
}

// The LK launch fields klt_lk_params decides: window, criteria (A.2: OpenCV's clamps) and eps2 brackets, flags, threshold
void set_lk_params(LKLaunch& L, const klt_lk_params* p)
{
    L.win_w = p->win_w; L.win_h = p->win_h;
    double eps;
    if ((p->crit_type & KLT_TERM_COUNT) == 0) L.max_count = 30;
    else L.max_count = p->crit_max_count < 0 ? 0 : (p->crit_max_count > 100 ? 100 : p->crit_max_count);
    if ((p->crit_type & KLT_TERM_EPS) == 0) eps = 0.01;
    else eps = p->crit_eps < 0. ? 0. : (p->crit_eps > 10. ? 10. : p->crit_eps);
    L.eps2 = eps * eps;
    L.flags = p->flags;
    L.min_eig_thr = (float)p->min_eig_threshold;
    if (L.eps2 >= 1e-30 && L.eps2 <= 1e30) {
        L.eps2_lo = std::nextafterf((float)(L.eps2 * (1.0 - 1.0 / 1048576.0)), -1.f);
        L.eps2_hi = std::nextafterf((float)(L.eps2 * (1.0 + 1.0 / 1048576.0)), 3.0e38f);
    } else {
        L.eps2_lo = -1.f;
        L.eps2_hi = __builtin_inff();
    }
}

}  // namespace

extern "C" {

int klt_version(void) { return KLT_B200_VERSION; }

const char* klt_status_string(klt_status s)
{
    switch (s) {
        case KLT_OK: return "ok";
        case KLT_ERR_INVALID_ARG: return "invalid argument (cv2 would raise an assertion error)";
        case KLT_ERR_UNSUPPORTED: return "valid for OpenCV but outside libklt_b200 limits";
        case KLT_ERR_NO_DEVICE: return "no sm_100 CUDA device available (there is no CPU fallback)";
        case KLT_ERR_OUT_OF_MEMORY: return "out of memory";
        case KLT_ERR_INTERNAL: return "internal error";
        default: return s > 0 ? cudaGetErrorString((cudaError_t)s) : "unknown status";
    }
}

klt_status klt_create(int device, klt_ctx** out)
{
    if (!out) return KLT_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return KLT_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    KLT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return KLT_ERR_NO_DEVICE;  // the fatbin holds sm_100a SASS only
    DeviceGuard guard(device);
    if (guard.err != cudaSuccess) return (klt_status)guard.err;
    klt_ctx* ctx = new (std::nothrow) klt_ctx();
    if (!ctx) return KLT_ERR_OUT_OF_MEMORY;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    std::snprintf(ctx->name, sizeof(ctx->name), "%s", prop.name);
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev2, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
        delete ctx;
        return (klt_status)e;
    }
    klt_status s = lk_init(device);
    if (s != KLT_OK) { cudaStreamDestroy(ctx->stream); cudaStreamDestroy(ctx->stream2); cudaEventDestroy(ctx->ev2); delete ctx; return s; }
    *out = ctx;
    return KLT_OK;
}

klt_status klt_destroy(klt_ctx* ctx)
{
    if (!ctx) return KLT_OK;
    DeviceGuard guard(ctx->device);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
    if (ctx->stream2) { cudaStreamSynchronize(ctx->stream2); cudaStreamDestroy(ctx->stream2); }
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    if (ctx->stager) { ctx->stager->shutdown(); delete ctx->stager; ctx->stager = nullptr; }
    if (ctx->d_ws) cudaFree(ctx->d_ws);
    if (ctx->h_ws) cudaFreeHost(ctx->h_ws);
    if (ctx->h_in) cudaFreeHost(ctx->h_in);
    if (ctx->h_step) cudaFreeHost(ctx->h_step);
    if (ctx->d_hash) cudaFree(ctx->d_hash);
    cudaDeviceSynchronize();   // caller streams that used the work lists may be gone already
    for (auto& sc : ctx->pyr_scratch) cudaFree(sc.cnt);
    for (auto& t : ctx->bilateral_tabs) cudaFree(t.d_tab);
    delete ctx;
    return KLT_OK;
}

klt_status klt_device_info(klt_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, char* name, int name_len)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (name && name_len > 0) std::snprintf(name, (size_t)name_len, "%s", ctx->name);
    return KLT_OK;
}

klt_status klt_host_alloc(void** ptr, int64_t bytes)
{
    if (!ptr || bytes <= 0) return KLT_ERR_INVALID_ARG;
    cudaError_t e = cudaMallocHost(ptr, (size_t)bytes);
    if (e != cudaSuccess) { *ptr = nullptr; return cuda_status(e); }
    return KLT_OK;
}

klt_status klt_host_free(void* ptr)
{
    if (!ptr) return KLT_OK;
    KLT_CUDA(cudaFreeHost(ptr));
    return KLT_OK;
}

klt_status klt_pyr_plan(int w, int h, int win_w, int win_h, int max_level, int batch, klt_pyr_layout* out)
{
    if (!out || w <= 0 || h <= 0 || win_w <= 2 || win_h <= 2 || max_level < 0 || batch <= 0) return KLT_ERR_INVALID_ARG;
    std::memset(out, 0, sizeof(*out));
    out->batch = batch;
    out->level[0].w = w;
    out->level[0].h = h;
    out->level[0].pitch = w;                       // caller overrides with the real image pitch
    out->level[0].batch_stride = (int64_t)w * h;   // idem
    int top = 0;
    int64_t off = 0;
    int lw = w, lh = h;
    while (top < max_level && top + 1 < KLT_MAX_LEVELS) {
        const int nw = (lw + 1) / 2, nh = (lh + 1) / 2;
        if (nw <= win_w || nh <= win_h) break;  // SURVEY.md A.2
        ++top;
        klt_level& L = out->level[top];
        L.w = nw; L.h = nh;
        L.pitch = (int64_t)align_up((size_t)nw, 32);
        L.batch_stride = (int64_t)align_up((size_t)(L.pitch * nh), 256);
        L.offset = off;
        off += L.batch_stride * batch;
        lw = nw; lh = nh;
    }
    out->top = top;
    out->bytes = off;
    return KLT_OK;
}

klt_status klt_pyr_down(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_batch_stride,
                        uint8_t* d_dst, int64_t dst_pitch, int64_t dst_batch_stride, int batch, void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return pyr_down_launch(d_src, w, h, src_pitch, src_batch_stride, d_dst, dst_pitch, dst_batch_stride, batch,
                           ctx->sm_count, (cudaStream_t)stream);
}

klt_status klt_pyr_build(klt_ctx* ctx, const uint8_t* d_img, const klt_pyr_layout* layout, uint8_t* d_pyr,
                         int first_item, int n_items, void* stream)
{
    if (!ctx || !d_img) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    klt_status s = check_layout(layout);
    if (s != KLT_OK) return s;
    if (layout->top > 0 && !d_pyr) return KLT_ERR_INVALID_ARG;
    if (n_items <= 0) { first_item = 0; n_items = layout->batch; }
    if (first_item < 0 || first_item + n_items > layout->batch) return KLT_ERR_INVALID_ARG;
    for (int l = 0; l < layout->top; ++l)
        if (layout->level[l + 1].w != (layout->level[l].w + 1) / 2 || layout->level[l + 1].h != (layout->level[l].h + 1) / 2) return KLT_ERR_INVALID_ARG;
    return pyr_build(ctx, d_img, layout, d_pyr, first_item, n_items, (cudaStream_t)stream);
}

klt_status klt_lk_track(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                        int prev_first, int next_first, int pair_stride, int n_pairs,
                        const float* d_prev_pts, float* d_next_pts, uint8_t* d_status, float* d_err,
                        int32_t* d_iters, int n_per_pair, const klt_lk_params* params, void* stream)
{
    if (!ctx || !params || !d_prev_img || !d_next_img || n_per_pair < 0 || n_pairs < 0) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    klt_status s = check_layout(layout);
    if (s != KLT_OK) return s;
    if (pair_stride < 1 || prev_first < 0 || next_first < 0) return KLT_ERR_INVALID_ARG;
    if (n_pairs > 0 && ((int64_t)prev_first + (int64_t)(n_pairs - 1) * pair_stride >= layout->batch ||
                        (int64_t)next_first + (int64_t)(n_pairs - 1) * pair_stride >= layout->batch))
        return KLT_ERR_INVALID_ARG;
    if (layout->top > 0 && (!d_prev_pyr || !d_next_pyr)) return KLT_ERR_INVALID_ARG;
    if (params->win_w <= 2 || params->win_h <= 2) return KLT_ERR_INVALID_ARG;
    if (n_per_pair == 0 || n_pairs == 0) return KLT_OK;
    if (!d_prev_pts || !d_next_pts || !d_status || !d_err) return KLT_ERR_INVALID_ARG;
    LKLaunch L;
    make_view(layout, d_prev_img, d_prev_pyr, prev_first, pair_stride, L.prev);
    make_view(layout, d_next_img, d_next_pyr, next_first, pair_stride, L.next);
    L.prev_pts = d_prev_pts; L.next_pts = d_next_pts; L.status = d_status; L.err = d_err; L.iters = d_iters;
    L.n_per_pair = n_per_pair;
    L.batch = n_pairs;
    set_lk_params(L, params);
    return lk_launch(L, ctx->sm_count, (cudaStream_t)stream);
}

}  // extern "C"

namespace {

// Shared worker of the host-pointer entry points: upload the pair, build both pyramids (one launch per level for the
// two images), track.  bidir: run the reference's second call (same direction, started from the forward result) and the
// bidirectional-error / bounds filter on the device as well -- one upload and one pyramid build for the whole step.
// reverse (with bidir): the second call runs from the new image back into the old one instead (klt_track_fb_host).
klt_status track_host(klt_ctx* ctx, const uint8_t* prev_img, int64_t prev_pitch, const uint8_t* next_img, int64_t next_pitch,
                      int w, int h, const float* prev_pts, float* next_pts, uint8_t* status, float* err, int n,
                      int max_level, const klt_lk_params* params, int* top_level_out, bool bidir, float max_bidir_error,
                      uint8_t* keep, float* bidir_err, bool reverse)
{
    if (!ctx || !params || !prev_img || !next_img || w <= 0 || h <= 0 || n < 0 || max_level < 0) return KLT_ERR_INVALID_ARG;
    if (prev_pitch < w || next_pitch < w) return KLT_ERR_INVALID_ARG;
    if (n > 0 && (!prev_pts || !next_pts || !status || !err)) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    // both images form a batch of 2 so that every pyramid level is ONE launch for the pair
    klt_pyr_layout lay;
    klt_status s = klt_pyr_plan(w, h, params->win_w, params->win_h, max_level, 2, &lay);
    if (s != KLT_OK) return s;
    if (top_level_out) *top_level_out = lay.top;
    if (n == 0) return KLT_OK;
    const size_t ipitch = align_up((size_t)w, 128);
    const size_t ibytes = align_up(ipitch * (size_t)h, 256);
    if (ipitch > 0x7fffffff) return KLT_ERR_INVALID_ARG;   // the kernels take 32-bit pitches (check_layout)
    lay.level[0].pitch = (int64_t)ipitch;
    lay.level[0].batch_stride = (int64_t)ibytes;
    const size_t off_img = 0;
    const size_t off_pyr = off_img + 2 * ibytes;
    const size_t off_pts = off_pyr + align_up((size_t)lay.bytes, 256);
    const size_t pts_bytes = align_up((size_t)n * 8, 256);
    const size_t off_out = off_pts + pts_bytes;                 // nextPts | err | [bidir err] | status | [keep], one D2H copy
    const size_t out_bytes = (size_t)n * 8 + (size_t)n * 4 + (bidir ? (size_t)n * 4 : 0) + (size_t)n + (bidir ? (size_t)n : 0);
    const size_t off_p0r = off_out + align_up(out_bytes, 256);  // second-call result (bidir only)
    // raw landing zone: each image arrives as ONE contiguous DMA in the caller's own row pitch, re-pitched on the device
    const size_t off_raw = off_p0r + (bidir ? pts_bytes : 0);
    const size_t raw_prev = raw_span(prev_pitch, w, h);
    const size_t raw_next = raw_span(next_pitch, w, h);
    const bool linear = near_contiguous(raw_prev, w, h) && near_contiguous(raw_next, w, h);
    const size_t raw_slot = linear ? align_up((raw_prev > raw_next ? raw_prev : raw_next) + 32, 256) : 0;
    // ---- pyramid reuse across calls: the images are hashed on the device while they are re-pitched; an item whose hash
    // equals that of the previous call (same geometry, workspace untouched since) keeps its pyramid.  The reference's four
    // calls per frame pass the same pair (extractor.py:44,45,65,66), so three of four builds go.
    const long long key[7] = {1, w, h, params->win_w, params->win_h, lay.top, (long long)ipitch};
    bool valid_prev = false;
    s = claim_device_ws(ctx, off_raw + 2 * raw_slot, key, &valid_prev);
    if (s != KLT_OK) return s;
    s = ensure_host_ws(ctx, align_up(out_bytes, 256));
    if (s != KLT_OK) return s;
    uint8_t* d = ctx->d_ws;
    cudaStream_t st = ctx->stream;
    // Hashing costs 2.4 us per call, a skipped build saves 7: it is switched on only while the caller keeps passing the same
    // two arrays (the first repeat builds and records the hashes, the following ones skip)
    const bool same_arrays = ctx->last_imgs[0] == prev_img && ctx->last_imgs[1] == next_img && ctx->last_pitch[0] == prev_pitch &&
                             ctx->last_pitch[1] == next_pitch;
    ctx->last_imgs[0] = prev_img; ctx->last_imgs[1] = next_img; ctx->last_pitch[0] = prev_pitch; ctx->last_pitch[1] = next_pitch;
    const bool hashing = linear && lay.top >= 2 && same_arrays;
    unsigned* h_new = nullptr;
    PyrReuse reuse = {nullptr, nullptr, nullptr, nullptr, 0u};
    if (hashing) {
        if (!ctx->d_hash) {
            KLT_CUDA(cudaMalloc(&ctx->d_hash, 32 * sizeof(unsigned)));
            KLT_CUDA(cudaMemset(ctx->d_hash, 0, 32 * sizeof(unsigned)));
            KLT_CUDA(cudaDeviceSynchronize());   // the memset is not ordered with the context's non-blocking streams
        }
        if (!valid_prev) KLT_CUDA(cudaMemsetAsync(ctx->d_hash, 0, 12 * sizeof(unsigned), st));   // slots may hold leftovers
        const unsigned k = (unsigned)(ctx->reuse_call % 3);
        h_new = ctx->d_hash + 4 * k;
        reuse.hash_new = h_new;
        reuse.hash_old = ctx->d_hash + 4 * ((k + 2) % 3);
        reuse.hash_clear = ctx->d_hash + 4 * ((k + 1) % 3);
        reuse.skipped = reinterpret_cast<unsigned long long*>(ctx->d_hash + 16);
        reuse.mask = valid_prev ? 3u : 0u;
    }
    const auto t0 = Clock::now();
    // The two image copies go out on two streams so that both DMA engines work and the fixed latency of one copy
    // hides behind the other (measured: zero-copy reads by the SMs are slower than the DMA engines for this size).
    cudaStream_t st2 = ctx->stream2;
    if (linear) {
        // Pageable inputs (what the un-edited reference passes) are staged through the context's pinned landing zone by
        // the calling thread and the helper threads; the DMA of the next image runs while the previous image is staged.
        const uint8_t* src_next = next_img;
        const uint8_t* src_prev = prev_img;
        const float* src_pts = prev_pts;
        // (an error return between the two halves must not leave helpers reading the caller's buffers)
        struct StageGuard {
            klt_ctx::Stager* s; bool done0 = false, done1 = false;
            void finish(int job) { if (s && !(job ? done1 : done0)) { s->finish_job(job); (job ? done1 : done0) = true; } }
            ~StageGuard() { finish(0); finish(1); }
        } stage_guard{nullptr};
        if (raw_prev + raw_next >= (256u << 10) && (is_pageable(prev_img) || is_pageable(next_img))) {
            const size_t in_slot = align_up(std::max(raw_prev, raw_next), 256);
            const size_t in_pts = align_up((size_t)n * 8, 256);
            s = ensure_host_in(ctx, 2 * in_slot + in_pts);
            if (s != KLT_OK) return s;
            stage_guard.s = stage_pageable(ctx, src_next, raw_next, src_prev, raw_prev, in_slot);
            if (stage_guard.s) {
                std::memcpy(ctx->h_in + 2 * in_slot, prev_pts, (size_t)n * 8);
                src_pts = reinterpret_cast<const float*>(ctx->h_in + 2 * in_slot);
            }
        }
        stage_guard.finish(0);
        KLT_CUDA(cudaMemcpyAsync(d + off_raw + raw_slot, src_next, raw_next, cudaMemcpyHostToDevice, st2));
        KLT_CUDA(cudaEventRecord(ctx->ev2, st2));
        KLT_CUDA(cudaMemcpyAsync(d + off_pts, src_pts, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        stage_guard.finish(1);
        KLT_CUDA(cudaMemcpyAsync(d + off_raw, src_prev, raw_prev, cudaMemcpyHostToDevice, st));
        KLT_CUDA(cudaStreamWaitEvent(st, ctx->ev2, 0));
        if (prev_pitch == next_pitch) {
            s = repitch_launch(d + off_raw, prev_pitch, (long long)raw_slot, d + off_img, (long long)ipitch, (long long)ibytes, w, h, 2, st, h_new);
        } else {
            s = repitch_launch(d + off_raw, prev_pitch, 0, d + off_img, (long long)ipitch, (long long)ibytes, w, h, 1, st, h_new);
            if (s == KLT_OK)
                s = repitch_launch(d + off_raw + raw_slot, next_pitch, 0, d + off_img + ibytes, (long long)ipitch, (long long)ibytes, w, h, 1, st,
                                   h_new ? h_new + 2 : nullptr);
        }
        if (s != KLT_OK) return s;
    } else {
        KLT_CUDA(cudaMemcpy2DAsync(d + off_img, ipitch, prev_img, (size_t)prev_pitch, (size_t)w, (size_t)h, cudaMemcpyHostToDevice, st));
        KLT_CUDA(cudaMemcpy2DAsync(d + off_img + ibytes, ipitch, next_img, (size_t)next_pitch, (size_t)w, (size_t)h, cudaMemcpyHostToDevice, st));
        KLT_CUDA(cudaMemcpyAsync(d + off_pts, prev_pts, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    }
    float* d_next = reinterpret_cast<float*>(d + off_out);
    float* d_err = reinterpret_cast<float*>(d + off_out + (size_t)n * 8);
    float* d_bidir = reinterpret_cast<float*>(d + off_out + (size_t)n * 12);
    const size_t o_status = (size_t)n * (bidir ? 16 : 12);
    uint8_t* d_status = d + off_out + o_status;
    uint8_t* d_keep = d_status + n;
    if (params->flags & KLT_OPTFLOW_USE_INITIAL_FLOW)
        KLT_CUDA(cudaMemcpyAsync(d_next, next_pts, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    const auto t1 = Clock::now();
    if (trace_on()) cudaStreamSynchronize(st);
    const auto t1s = Clock::now();
    bool reuse_armed = false;
    s = pyr_build(ctx, d + off_img, &lay, d + off_pyr, 0, 2, st, hashing ? &reuse : nullptr, &reuse_armed);
    if (s != KLT_OK) return s;
    // the pair lives in one batch-2 pyramid: prev = item 0, next = item 1
    LKLaunch L;
    make_view(&lay, d + off_img, d + off_pyr, 0, 1, L.prev);
    make_view(&lay, d + off_img, d + off_pyr, 1, 1, L.next);
    // results: the kernel writes its 13 bytes per point straight into the context's page-locked staging buffer (mapped
    // into the device address space), so no D2H copy is queued -- unless nextPts is also an input (initial flow)
    const bool direct = !bidir && !(params->flags & KLT_OPTFLOW_USE_INITIAL_FLOW) && ctx->h_ws_dev != nullptr;
    if (direct) {
        d_next = reinterpret_cast<float*>(ctx->h_ws_dev);
        d_err = reinterpret_cast<float*>(ctx->h_ws_dev + (size_t)n * 8);
        d_status = ctx->h_ws_dev + (size_t)n * 12;
    }
    L.prev_pts = reinterpret_cast<const float*>(d + off_pts);
    L.next_pts = d_next; L.status = d_status; L.err = d_err; L.iters = nullptr;
    L.n_per_pair = n; L.batch = 1;
    set_lk_params(L, params);
    s = lk_launch(L, ctx->sm_count, st);
    if (s != KLT_OK) return s;
    if (bidir) {
        // second call of the reference (extractor.py:45,66): same image pair, prevPts = the forward result.  The
        // reference discards its status / err, so they land in the keep / bidir slots that the filter overwrites next.
        LKLaunch L2 = L;
        if (reverse) std::swap(L2.prev, L2.next);
        L2.prev_pts = d_next;
        L2.next_pts = reinterpret_cast<float*>(d + off_p0r);
        L2.status = d_keep;                       // overwritten by the filter below
        L2.err = d_bidir;                         // idem
        s = lk_launch(L2, ctx->sm_count, st);
        if (s != KLT_OK) return s;
        s = track_filter_launch(L.prev_pts, d_next, L2.next_pts, n, max_bidir_error, w, h, d_keep, d_bidir, st);
        if (s != KLT_OK) return s;
    }
    const auto t2 = Clock::now();
    if (trace_on()) cudaStreamSynchronize(st);
    const auto t2s = Clock::now();
    if (!direct) KLT_CUDA(cudaMemcpyAsync(ctx->h_ws, d + off_out, out_bytes, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    const auto t3 = Clock::now();
    if (trace_on())
        std::fprintf(stderr, "[klt trace] h2d enqueue %.1f us, h2d done +%.1f us, kernels enqueue %.1f us, kernels done +%.1f us, d2h+sync %.1f us\n",
                     us(t0, t1), us(t1, t1s), us(t1s, t2), us(t2, t2s), us(t2s, t3));
    if (reuse_armed) {   // the pyramids in the workspace now belong to the images of this call
        std::memcpy(ctx->reuse_key, key, sizeof(key));
        ++ctx->reuse_call;
    }
    std::memcpy(next_pts, ctx->h_ws, (size_t)n * 8);
    std::memcpy(err, ctx->h_ws + (size_t)n * 8, (size_t)n * 4);
    std::memcpy(status, ctx->h_ws + o_status, (size_t)n);
    if (bidir) {
        std::memcpy(bidir_err, ctx->h_ws + (size_t)n * 12, (size_t)n * 4);
        std::memcpy(keep, ctx->h_ws + o_status + n, (size_t)n);
    }
    return KLT_OK;
}

}  // namespace

extern "C" {

klt_status klt_calc_optical_flow_pyr_lk_host(klt_ctx* ctx, const uint8_t* prev_img, int64_t prev_pitch,
                                             const uint8_t* next_img, int64_t next_pitch, int w, int h,
                                             const float* prev_pts, float* next_pts, uint8_t* status, float* err,
                                             int n, int max_level, const klt_lk_params* params, int* top_level_out)
{
    return track_host(ctx, prev_img, prev_pitch, next_img, next_pitch, w, h, prev_pts, next_pts, status, err, n, max_level,
                      params, top_level_out, false, 0.f, nullptr, nullptr, false);
}

klt_status klt_track_bidirectional_host(klt_ctx* ctx, const uint8_t* prev_img, int64_t prev_pitch,
                                        const uint8_t* next_img, int64_t next_pitch, int w, int h,
                                        const float* prev_pts, int n, int max_level, const klt_lk_params* params,
                                        float max_bidir_error, float* next_pts, uint8_t* status, float* err,
                                        uint8_t* keep, float* bidir_err)
{
    if (n > 0 && (!keep || !bidir_err)) return KLT_ERR_INVALID_ARG;
    if (params && (params->flags & KLT_OPTFLOW_USE_INITIAL_FLOW)) return KLT_ERR_INVALID_ARG;   // the reference passes nextPts = None
    return track_host(ctx, prev_img, prev_pitch, next_img, next_pitch, w, h, prev_pts, next_pts, status, err, n, max_level,
                      params, nullptr, true, max_bidir_error, keep, bidir_err, false);
}

klt_status klt_track_fb_host(klt_ctx* ctx, const uint8_t* prev_img, int64_t prev_pitch, const uint8_t* next_img, int64_t next_pitch,
                             int w, int h, const float* prev_pts, int n, int max_level, const klt_lk_params* params,
                             float max_bidir_error, float* next_pts, uint8_t* status, float* err, uint8_t* keep, float* bidir_err)
{
    if (n > 0 && (!keep || !bidir_err)) return KLT_ERR_INVALID_ARG;
    if (params && (params->flags & KLT_OPTFLOW_USE_INITIAL_FLOW)) return KLT_ERR_INVALID_ARG;   // no start positions here
    return track_host(ctx, prev_img, prev_pitch, next_img, next_pitch, w, h, prev_pts, next_pts, status, err, n, max_level,
                      params, nullptr, true, max_bidir_error, keep, bidir_err, true);
}

klt_status klt_track_filter(klt_ctx* ctx, const float* d_p0, const float* d_p1, const float* d_p0r, int64_t n,
                            float max_bidir_error, int w, int h, uint8_t* d_keep, float* d_bidir_err, void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return track_filter_launch(d_p0, d_p1, d_p0r, (long long)n, max_bidir_error, w, h, d_keep, d_bidir_err, (cudaStream_t)stream);
}

klt_status klt_build_optical_flow_pyramid_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                                               int win_w, int win_h, int max_level, uint8_t* out,
                                               int64_t* level_offsets, int* top_out)
{
    if (!ctx || w <= 0 || h <= 0 || max_level < 0) return KLT_ERR_INVALID_ARG;
    klt_pyr_layout lay;
    klt_status s = klt_pyr_plan(w, h, win_w, win_h, max_level, 1, &lay);
    if (s != KLT_OK) return s;
    if (top_out) *top_out = lay.top;
    int64_t off = 0;
    for (int l = 0; l <= lay.top; ++l) {
        if (level_offsets) level_offsets[l] = off;
        off += (int64_t)lay.level[l].w * lay.level[l].h;
    }
    if (level_offsets) level_offsets[lay.top + 1] = off;
    if (!out) return KLT_OK;
    if (!img || pitch < w) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    const size_t ipitch = align_up((size_t)w, 128);
    const size_t ibytes = align_up(ipitch * (size_t)h, 256);
    if (ipitch > 0x7fffffff) return KLT_ERR_INVALID_ARG;   // the kernels take 32-bit pitches (check_layout)
    lay.level[0].pitch = (int64_t)ipitch;
    lay.level[0].batch_stride = (int64_t)ibytes;
    s = claim_device_ws(ctx, ibytes + (size_t)lay.bytes, nullptr, nullptr);
    if (s != KLT_OK) return s;
    uint8_t* d = ctx->d_ws;
    cudaStream_t st = ctx->stream;
    KLT_CUDA(cudaMemcpy2DAsync(d, ipitch, img, (size_t)pitch, (size_t)w, (size_t)h, cudaMemcpyHostToDevice, st));
    s = pyr_build(ctx, d, &lay, d + ibytes, 0, 1, st);
    if (s != KLT_OK) return s;
    int64_t o = 0;
    for (int l = 0; l <= lay.top; ++l) {
        const klt_level& L = lay.level[l];
        const uint8_t* src = (l == 0) ? d : d + ibytes + L.offset;
        KLT_CUDA(cudaMemcpy2DAsync(out + o, (size_t)L.w, src, (size_t)L.pitch, (size_t)L.w, (size_t)L.h, cudaMemcpyDeviceToHost, st));
        o += (int64_t)L.w * L.h;
    }
    KLT_CUDA(cudaStreamSynchronize(st));
    return KLT_OK;
}

// ---- Shi-Tomasi corner detection (SURVEY.md s8f rank 2; kernels in klt_corners.cu) -----------------------------------

int64_t klt_corner_ws_bytes(int w, int h, int batch)
{
    if (w < 1 || h < 1 || batch < 1) return 0;
    return (int64_t)corners_ws_bytes(w, h, batch);
}

klt_status klt_corner_min_eigen_val(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride,
                                    int batch, int block_size, float* d_eig, int64_t eig_pitch, int64_t eig_batch_stride,
                                    const uint8_t* d_mask, int64_t mask_pitch, int64_t mask_batch_stride, uint32_t* d_max,
                                    void* d_ws, int64_t ws_bytes, void* stream)
{
    if (!ctx || !d_img || !d_eig || !d_ws || pitch < w || eig_pitch < w) return KLT_ERR_INVALID_ARG;
    if (w < 1 || h < 1 || batch < 1 || block_size < 1) return KLT_ERR_INVALID_ARG;
    if (ws_bytes < (int64_t)corners_ws_bytes(w, h, batch) || ((uintptr_t)d_ws & 255)) return KLT_ERR_INVALID_ARG;
    if (d_mask && mask_pitch < w) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return corner_min_eig_launch(d_img, pitch, batch_stride, w, h, batch, block_size, d_eig, eig_pitch, eig_batch_stride,
                                 d_mask, mask_pitch, mask_batch_stride, d_max, d_ws, (cudaStream_t)stream);
}

klt_status klt_corner_candidates(klt_ctx* ctx, const float* d_eig, int64_t eig_pitch, int64_t eig_batch_stride, int w, int h,
                                 int batch, const uint8_t* d_mask, int64_t mask_pitch, int64_t mask_batch_stride,
                                 const uint32_t* d_max, double quality_level, uint64_t* d_keys, int64_t keys_batch_stride,
                                 int capacity, uint32_t* d_count, void* stream)
{
    if (!ctx || !d_eig || !d_max || !d_keys || !d_count || eig_pitch < w) return KLT_ERR_INVALID_ARG;
    if (d_mask && mask_pitch < w) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return corner_candidates_launch(d_eig, eig_pitch, eig_batch_stride, w, h, batch, d_mask, mask_pitch, mask_batch_stride,
                                    d_max, quality_level, reinterpret_cast<unsigned long long*>(d_keys), keys_batch_stride,
                                    capacity, d_count, (cudaStream_t)stream);
}

static klt_status select_corners(uint64_t* keys, int64_t n_keys, bool sorted, int w, int h, int max_corners, double min_distance,
                                 float* corners, int capacity, int* n_out)
{
    if (!n_out || n_keys < 0 || (n_keys > 0 && !keys) || w < 1 || h < 1 || max_corners < 0 || !(min_distance >= 0) ||
        capacity < 0 || (capacity > 0 && !corners))
        return KLT_ERR_INVALID_ARG;
    *n_out = 0;
    // strongest first; equal values: the later pixel in raster order first (OpenCV sorts pointers into the eigenvalue image with
    // "*a > *b, then a > b") -- both are the descending order of the 64-bit key
    if (sorted) {
        // the device already sorted them
    } else if (n_keys < 256) {
        std::sort(keys, keys + n_keys, std::greater<uint64_t>());
    } else {
        // LSD radix sort on the value half (3 passes of 11 / 11 / 10 bits, descending, stable), then the (rare) runs
        // of equal values are ordered by descending index
        std::vector<uint64_t> tmp;
        try { tmp.resize((size_t)n_keys); } catch (const std::bad_alloc&) { return KLT_ERR_OUT_OF_MEMORY; }
        uint64_t* src = keys;
        uint64_t* dst = tmp.data();
        const int shift[3] = {32, 43, 54}, bits[3] = {11, 11, 10};
        for (int p = 0; p < 3; ++p) {
            const unsigned nb = 1u << bits[p], msk = nb - 1u;
            unsigned hist[2048] = {0};
            for (int64_t i = 0; i < n_keys; ++i) ++hist[msk - (unsigned)((src[i] >> shift[p]) & msk)];
            unsigned run = 0;
            for (unsigned d = 0; d < nb; ++d) { const unsigned c = hist[d]; hist[d] = run; run += c; }
            for (int64_t i = 0; i < n_keys; ++i) dst[hist[msk - (unsigned)((src[i] >> shift[p]) & msk)]++] = src[i];
            std::swap(src, dst);
        }
        // three passes: the result is in tmp
        for (int64_t i = 0; i < n_keys;) {
            int64_t j = i + 1;
            while (j < n_keys && (src[j] >> 32) == (src[i] >> 32)) ++j;
            if (j - i > 1) std::sort(src + i, src + j, std::greater<uint64_t>());
            i = j;
        }
        std::memcpy(keys, src, (size_t)n_keys * 8);
    }
    int nc = 0;
    auto emit = [&](int x, int y) {
        if (nc < capacity) { corners[2 * nc] = (float)x; corners[2 * nc + 1] = (float)y; }
        ++nc;
        return max_corners > 0 && nc == max_corners;
    };
    if (min_distance >= 1) {
        // G.8: grid of cells of size cvRound(minDistance); a candidate is dropped if an accepted corner in the 3 x 3
        // neighbouring cells is closer than minDistance
        const int cell = (int)std::lrint(min_distance);
        const int gw = (w + cell - 1) / cell, gh = (h + cell - 1) / cell;
        const double md2 = min_distance * min_distance;
        const double md2c = std::ceil(md2);   // squared pixel distances are integers: d2 < md2  <=>  d2 < ceil(md2)
        const long long md2i = md2c < 9.0e18 ? (long long)md2c : (long long)9.0e18;
        // x / cell for 16-bit x by multiplication: exact since x * (cell - 1) < 2^32
        const uint64_t magic = cell > 1 ? ((1ull << 32) + (uint64_t)cell - 1) / (uint64_t)cell : 0;
        if ((size_t)(gw + 2) * (gh + 2) <= (1u << 20)) {
            // Fast path: a padded grid (no clamping) of per-cell counters and up to 4 inline corners per cell -- accepted
            // corners are >= minDistance apart and a cell is at most minDistance + 0.5 wide, so 4 is never exceeded (checked).
            // A candidate first reads the 3 x 3 counters (three 3-byte reads); most candidates have empty neighbourhoods
            // late in the list or find their conflict in the first occupied cell.
            struct Cell { unsigned short x[4], y[4]; };   // keys carry 16-bit unsigned coordinates (w, h <= 65535)
            const int gw2 = gw + 2;
            const size_t ncell = (size_t)gw2 * (gh + 2);
            thread_local std::vector<unsigned char> cnt_buf;
            thread_local std::vector<Cell> cell_buf;
            try {
                cnt_buf.assign(ncell + 4, 0);
                if (cell_buf.size() < ncell) cell_buf.resize(ncell);
            } catch (const std::bad_alloc&) { return KLT_ERR_OUT_OF_MEMORY; }
            unsigned char* cnt = cnt_buf.data();
            Cell* cells = cell_buf.data();
            for (int64_t i = 0; i < n_keys; ++i) {
                const int x = (int)(keys[i] & 0xffffu), y = (int)((keys[i] >> 16) & 0xffffu);
                if (y >= h || x >= w) return KLT_ERR_INVALID_ARG;
                const int xc = cell > 1 ? (int)(((uint64_t)x * magic) >> 32) : x, yc = cell > 1 ? (int)(((uint64_t)y * magic) >> 32) : y;
                const size_t c0 = (size_t)yc * gw2 + xc;            // padded index of cell (yc - 1, xc - 1)
                bool good = true;
                for (int ry = 0; ry < 3 && good; ++ry) {
                    const size_t row = c0 + (size_t)ry * gw2;
                    if (!(cnt[row] | cnt[row + 1] | cnt[row + 2])) continue;
                    for (int rx = 0; rx < 3 && good; ++rx) {
                        const int m = cnt[row + rx];
                        const Cell& cl = cells[row + rx];
                        for (int j = 0; j < m; ++j) {
                            const long long dx = x - (int)cl.x[j], dy = y - (int)cl.y[j];
                            if (dx * dx + dy * dy < md2i) { good = false; break; }
                        }
                    }
                }
                if (!good) continue;
                const size_t cc = c0 + gw2 + 1;
                if (cnt[cc] >= 4) return KLT_ERR_INTERNAL;
                cells[cc].x[cnt[cc]] = (unsigned short)x; cells[cc].y[cnt[cc]] = (unsigned short)y; ++cnt[cc];
                if (emit(x, y)) break;
            }
            *n_out = nc;
            return KLT_OK;
        }
        // accepted corners: per-cell singly linked lists in flat arrays (scratch kept per thread across calls)
        const size_t max_acc = (size_t)((max_corners > 0 && max_corners < n_keys) ? max_corners : n_keys);
        thread_local std::vector<int> scratch;
        try {
            scratch.resize((size_t)gw * gh + 3 * max_acc + 1);
        } catch (const std::bad_alloc&) { return KLT_ERR_OUT_OF_MEMORY; }
        int* head = scratch.data();
        int* next = head + (size_t)gw * gh;
        int* ax = next + max_acc;
        int* ay = ax + max_acc;
        std::fill(head, head + (size_t)gw * gh, -1);
        int nacc = 0;
        for (int64_t i = 0; i < n_keys; ++i) {
            const int x = (int)(keys[i] & 0xffffu), y = (int)((keys[i] >> 16) & 0xffffu);
            if (y >= h || x >= w) return KLT_ERR_INVALID_ARG;
            const int xc = cell > 1 ? (int)(((uint64_t)x * magic) >> 32) : x, yc = cell > 1 ? (int)(((uint64_t)y * magic) >> 32) : y;
            const int x1 = std::max(0, xc - 1), y1 = std::max(0, yc - 1), x2 = std::min(gw - 1, xc + 1), y2 = std::min(gh - 1, yc + 1);
            bool good = true;
            for (int yy = y1; yy <= y2 && good; ++yy)
                for (int xx = x1; xx <= x2 && good; ++xx)
                    for (int j = head[(size_t)yy * gw + xx]; j >= 0; j = next[j]) {
                        const long long dx = x - ax[j], dy = y - ay[j];
                        if (dx * dx + dy * dy < md2i) { good = false; break; }
                    }
            if (!good) continue;
            ax[nacc] = x; ay[nacc] = y;
            next[nacc] = head[(size_t)yc * gw + xc];
            head[(size_t)yc * gw + xc] = nacc++;
            if (emit(x, y)) break;
        }
    } else {
        for (int64_t i = 0; i < n_keys; ++i) {
            if (emit((int)(keys[i] & 0xffffu), (int)((keys[i] >> 16) & 0xffffu))) break;
        }
    }
    *n_out = nc;
    return KLT_OK;
}

klt_status klt_select_corners_host(uint64_t* keys, int64_t n_keys, int w, int h, int max_corners, double min_distance,
                                   float* corners, int capacity, int* n_out)
{
    return select_corners(keys, n_keys, false, w, h, max_corners, min_distance, corners, capacity, n_out);
}

klt_status klt_corner_min_eigen_val_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, int block_size,
                                         float* eig)
{
    if (!ctx || !img || !eig || w < 1 || h < 1 || pitch < w || block_size < 1) return KLT_ERR_INVALID_ARG;
    if (block_size / 2 >= w || block_size / 2 >= h) return KLT_ERR_UNSUPPORTED;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    const size_t img_bytes = upload_bytes(pitch, w, h);
    const size_t eig_bytes = align_up((size_t)w * h * 4, 256);
    const size_t ws_bytes = (size_t)corners_ws_bytes(w, h, 1);
    klt_status s = claim_device_ws(ctx, img_bytes + eig_bytes + ws_bytes, nullptr, nullptr);
    if (s != KLT_OK) return s;
    uint8_t* d = ctx->d_ws;
    cudaStream_t st = ctx->stream;
    int64_t dpitch = 0;
    s = upload_u8(d, &dpitch, img, pitch, w, h, st);
    if (s != KLT_OK) return s;
    float* d_eig = reinterpret_cast<float*>(d + img_bytes);
    s = corner_min_eig_launch(d, dpitch, 0, w, h, 1, block_size, d_eig, w, 0, nullptr, 0, 0, nullptr, d + img_bytes + eig_bytes, st);
    if (s != KLT_OK) return s;
    KLT_CUDA(cudaMemcpyAsync(eig, d_eig, (size_t)w * h * 4, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    return KLT_OK;
}

// mask given by the caller (host image) or rasterised on the device from `points` (n_points >= 0 with mask == NULL and
// mask_radius >= 0: extractor.py:102-107)
static klt_status gftt_host_impl(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                                 const uint8_t* mask, int64_t mask_pitch, const float* points, int n_points, int mask_radius,
                                 int max_corners, double quality_level,
                                 double min_distance, int block_size, float* corners, int capacity, int* n_out)
{
    const bool from_points = mask_radius >= 0;
    if (from_points && (mask || n_points < 0 || (n_points > 0 && !points) || mask_radius > 127)) return mask_radius > 127 ? KLT_ERR_UNSUPPORTED : KLT_ERR_INVALID_ARG;
    if (!ctx || !img || !n_out || w < 1 || h < 1 || pitch < w || block_size < 1 || capacity < 0 || (capacity > 0 && !corners))
        return KLT_ERR_INVALID_ARG;
    if (!(quality_level > 0) || !(min_distance >= 0) || max_corners < 0) return KLT_ERR_INVALID_ARG;   // CV_Assert of goodFeaturesToTrack
    if (mask && mask_pitch < w) return KLT_ERR_INVALID_ARG;
    if (block_size / 2 >= w || block_size / 2 >= h || w > 65535 || h > 65535) return KLT_ERR_UNSUPPORTED;
    *n_out = 0;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    const size_t img_bytes = upload_bytes(pitch, w, h);
    const size_t pts_bytes = from_points ? align_up((size_t)n_points * 8 + 8, 256) : 0;
    const size_t mask_bytes = mask ? upload_bytes(mask_pitch, w, h) : (from_points ? align_up((size_t)w * h, 256) + pts_bytes : 0);
    const size_t eig_bytes = align_up((size_t)w * h * 4, 256);
    const size_t ws_bytes = (size_t)corners_ws_bytes(w, h, 1);
    // up to direct_cap sorted candidate keys land directly in the context's page-locked, device-mapped staging buffer
    const size_t n_px = (size_t)w * h;
    const size_t direct_cap = std::min<size_t>(n_px, 1u << 16);
    const size_t off_img = 0, off_mask = off_img + img_bytes, off_eig = off_mask + mask_bytes, off_ws = off_eig + eig_bytes;
    const size_t off_cnt = off_ws + ws_bytes, off_keys = off_cnt + 256 + 8192 * 4;   // max, count, ranks (zeroed per call)
    klt_status s = claim_device_ws(ctx, off_keys + (n_px + 1 + direct_cap) * 8, nullptr, nullptr);   // keys | header + sorted keys when not mapped
    if (s != KLT_OK) return s;
    s = ensure_host_ws(ctx, 8 + direct_cap * 8);
    if (s != KLT_OK) return s;
    uint8_t* d = ctx->d_ws;
    cudaStream_t st = ctx->stream, st2 = ctx->stream2;
    unsigned* d_max = reinterpret_cast<unsigned*>(d + off_cnt);
    unsigned* d_count = d_max + 1;
    KLT_CUDA(cudaMemsetAsync(d_max, 0, 256 + 8192 * 4, st));
    int64_t ipitch = 0, mpitch = 0;
    if (mask) {
        s = upload_u8(d + off_mask, &mpitch, mask, mask_pitch, w, h, st2);
        if (s != KLT_OK) return s;
        KLT_CUDA(cudaEventRecord(ctx->ev2, st2));
    } else if (from_points) {
        // tracked keypoints up (8 bytes each), discs rasterised on the device while the image is still in flight
        float* d_pts = reinterpret_cast<float*>(d + off_mask + align_up((size_t)w * h, 256));
        if (n_points > 0) KLT_CUDA(cudaMemcpyAsync(d_pts, points, (size_t)n_points * 8, cudaMemcpyHostToDevice, st2));
        mpitch = w;
        s = corner_mask_from_points_launch(d_pts, 0, nullptr, n_points, 1, mask_radius, w, h, d + off_mask, mpitch, 0, st2);
        if (s != KLT_OK) return s;
        KLT_CUDA(cudaEventRecord(ctx->ev2, st2));
    }
    s = upload_u8(d + off_img, &ipitch, img, pitch, w, h, st);
    if (s != KLT_OK) return s;
    if (mask || from_points) KLT_CUDA(cudaStreamWaitEvent(st, ctx->ev2, 0));
    const uint8_t* d_mask = (mask || from_points) ? d + off_mask : nullptr;
    float* d_eig = reinterpret_cast<float*>(d + off_eig);
    const auto t0 = Clock::now();
    if (trace_on()) cudaStreamSynchronize(st);
    const auto t1 = Clock::now();
    s = corner_min_eig_launch(d + off_img, ipitch, 0, w, h, 1, block_size, d_eig, w, 0, d_mask, mpitch, 0, d_max, d + off_ws, st);
    if (s != KLT_OK) return s;
    if (trace_on()) cudaStreamSynchronize(st);
    const auto t2 = Clock::now();
    // candidates -> device list (one slot per pixel: cannot overflow) -> sorted on the device -> written, with their
    // count, straight into the context's page-locked staging buffer (mapped into the device address space): no copy op
    unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(d + off_keys);
    s = corner_candidates_launch(d_eig, w, 0, w, h, 1, d_mask, mpitch, 0, d_max, quality_level, d_keys, 0, (int)n_px, d_count, st);
    if (s != KLT_OK) return s;
    const bool direct = ctx->h_ws_dev != nullptr;
    unsigned long long* d_out = direct ? reinterpret_cast<unsigned long long*>(ctx->h_ws_dev) : d_keys + n_px;
    s = corner_sort_launch(d_keys, 0, d_count, 1, reinterpret_cast<unsigned*>(d + off_cnt + 256), d_out, 0, (int)direct_cap, st);
    if (s != KLT_OK) return s;
    if (!direct) KLT_CUDA(cudaMemcpyAsync(ctx->h_ws, d_out, 8 + direct_cap * 8, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    const uint64_t header = *reinterpret_cast<const uint64_t*>(ctx->h_ws);
    const unsigned count = (unsigned)(header & 0xffffffffu);
    bool sorted = (header >> 32) & 1;
    uint64_t* h_keys = reinterpret_cast<uint64_t*>(ctx->h_ws) + 1;
    if (count > n_px) return KLT_ERR_INTERNAL;
    if (count > direct_cap) {
        // more candidates than the staging buffer holds (4K frames, plateaus): copy the whole unsorted list
        s = ensure_host_ws(ctx, 8 + (size_t)count * 8);   // may move the staging buffer; the device list is untouched
        if (s != KLT_OK) return s;
        h_keys = reinterpret_cast<uint64_t*>(ctx->h_ws) + 1;
        KLT_CUDA(cudaMemcpyAsync(h_keys, d_keys, (size_t)count * 8, cudaMemcpyDeviceToHost, st));
        KLT_CUDA(cudaStreamSynchronize(st));
        sorted = false;
    }
    const auto t3 = Clock::now();
    s = select_corners(h_keys, (int64_t)count, sorted, w, h, max_corners, min_distance, corners, capacity, n_out);
    if (trace_on())
        std::fprintf(stderr, "[klt trace] gftt: h2d done +%.1f us, eigenvalue kernels +%.1f us, candidates + sort + sync +%.1f us (%u candidates), host sort + selection %.1f us\n",
                     us(t0, t1), us(t1, t2), us(t2, t3), count, us(t3, Clock::now()));
    return s;
}

klt_status klt_good_features_to_track_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                                           const uint8_t* mask, int64_t mask_pitch, int max_corners, double quality_level,
                                           double min_distance, int block_size, float* corners, int capacity, int* n_out)
{
    return gftt_host_impl(ctx, img, pitch, w, h, mask, mask_pitch, nullptr, 0, -1, max_corners, quality_level, min_distance, block_size,
                          corners, capacity, n_out);
}

klt_status klt_good_features_to_track_points_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                                                  const float* points, int n_points, int mask_radius, int max_corners,
                                                  double quality_level, double min_distance, int block_size, float* corners,
                                                  int capacity, int* n_out)
{
    if (mask_radius < 0) return KLT_ERR_INVALID_ARG;
    return gftt_host_impl(ctx, img, pitch, w, h, nullptr, 0, points, n_points, mask_radius, max_corners, quality_level, min_distance,
                          block_size, corners, capacity, n_out);
}

klt_status klt_corner_mask_from_points(klt_ctx* ctx, const float* d_points, int n, int radius, int w, int h, uint8_t* d_mask,
                                       int64_t mask_pitch, void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return corner_mask_from_points_launch(d_points, 0, nullptr, n, 1, radius, w, h, d_mask, mask_pitch, 0, (cudaStream_t)stream);
}

// ---- grid detection: goodFeaturesToTrack per cell of a grid, for a batch of images --------------------------------------

namespace {

struct GridDetWs {
    size_t eig, cws, keys, thr, seg_count, n_sel, total;
};

GridDetWs grid_det_ws(int w, int h, int batch, int cells)
{
    GridDetWs o;
    const size_t px = (size_t)w * h, B = (size_t)batch, words = B * cells * 4;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off = align_up(off + bytes, 256); return at; };
    o.eig = take(B * px * 4);
    o.cws = take((size_t)corners_ws_bytes(w, h, batch));
    o.keys = take(B * px * 8);
    o.thr = take(words);
    o.seg_count = take(words);
    o.n_sel = take(words);
    o.total = off;
    return o;
}

}  // namespace

int64_t klt_good_features_to_track_grid_ws_bytes(int w, int h, int batch, int cols, int rows)
{
    if (w < 1 || h < 1 || batch < 1 || cols < 1 || rows < 1 || (int64_t)cols * rows > KLT_MAX_GRID_CELLS) return 0;
    return (int64_t)grid_det_ws(w, h, batch, cols * rows).total;
}

klt_status klt_good_features_to_track_grid(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride,
                                           int batch, int cols, int rows, int max_corners_per_cell, double quality_level,
                                           double min_distance, int block_size, const uint8_t* d_mask, int64_t mask_pitch,
                                           int64_t mask_batch_stride, float* d_corners, int32_t* d_counts, void* d_ws, int64_t ws_bytes,
                                           void* stream)
{
    if (!ctx || !d_img || !d_corners || !d_counts || !d_ws || w < 1 || h < 1 || batch < 1 || pitch < w) return KLT_ERR_INVALID_ARG;
    if (!(quality_level > 0) || !(min_distance >= 0) || max_corners_per_cell < 1 || block_size < 1) return KLT_ERR_INVALID_ARG;
    if (cols < 1 || rows < 1 || cols > w || rows > h || (d_mask && mask_pitch < w)) return KLT_ERR_INVALID_ARG;
    if ((int64_t)cols * rows > KLT_MAX_GRID_CELLS || w > 65535 || h > 65535 || batch > 21845) return KLT_ERR_UNSUPPORTED;
    const int G = cols * rows;
    const GridDetWs o = grid_det_ws(w, h, batch, G);
    if (ws_bytes < (int64_t)o.total || ((uintptr_t)d_ws & 255)) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* d = static_cast<uint8_t*>(d_ws);
    const long long px = (long long)w * h;
    float* d_eig = reinterpret_cast<float*>(d + o.eig);
    unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(d + o.keys);
    int* d_n_sel = reinterpret_cast<int*>(d + o.n_sel);
    klt_status s = corner_min_eig_launch(d_img, pitch, batch_stride, w, h, batch, block_size, d_eig, w, px, nullptr, 0, 0, nullptr, d + o.cws, st);
    if (s != KLT_OK) return s;
    s = corner_grid_detect_launch(d_eig, w, px, w, h, batch, d_mask, mask_pitch, mask_batch_stride, cols, rows, quality_level, min_distance,
                                  max_corners_per_cell, max_corners_per_cell, nullptr, nullptr, reinterpret_cast<float*>(d + o.thr),
                                  reinterpret_cast<unsigned*>(d + o.seg_count), d_n_sel, d_keys, px,
                                  reinterpret_cast<unsigned long long*>(d + o.cws), px, reinterpret_cast<unsigned*>(d_eig), px, st);
    if (s != KLT_OK) return s;
    return corner_grid_out_launch(d_keys, px, d_n_sel, w, h, batch, cols, rows, max_corners_per_cell, d_corners, d_counts, st);
}

// ---- the per-frame step for a batch of sequences ----------------------------------------------------------------------

}  // extern "C"

namespace {

// Device workspace of klt_frame_step_batch[_async], 256-byte aligned pieces.  The flag word (bad counts, for
// klt_frame_step_batch) and the block behind it (maximum eigenvalues, candidate counts, ranks of the key sort) are
// cleared by one memset.  Two regions are reused once their kernels are done with them: the corner scans' scratch (cws,
// about 36 bytes per pixel, free after col_scan_kernel) holds the radix sort's second key list (8 bytes per pixel), and
// the eigenvalue map (free after candidates_kernel) the selection bitmap of frames too large for shared memory.
struct StepWs {
    size_t p1, p0r, status, err, mask, eig, cws, surv, flag, max, count, rank, zero_end, keys, sorted, total;
};

constexpr int kStepSortCap = 8192;   // keys corner_sort_launch sorts per image (more: corner_radix_sort_launch sorts them)

StepWs step_ws(int w, int h, int batch, int n)
{
    StepWs o;
    const size_t B = (size_t)batch, px = (size_t)w * h, pts = B * (size_t)n;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off = align_up(off + bytes, 256); return at; };
    o.p1 = take(pts * 8);
    o.p0r = take(pts * 8);
    o.status = take(pts);
    o.err = take(pts * 4);
    o.mask = take(B * px);
    o.eig = take(B * px * 4);
    o.cws = take((size_t)corners_ws_bytes(w, h, batch));
    o.surv = off;
    o.flag = o.surv + B * 4;
    o.max = align_up(o.flag + 4, 16);
    o.count = o.max + B * 4;
    o.rank = align_up(o.count + B * 4, 16);
    o.zero_end = o.rank + B * kStepSortCap * 4;
    off = align_up(o.zero_end, 256);
    o.keys = take(B * px * 8);
    o.sorted = take(B * (1 + kStepSortCap) * 8);
    o.total = off;
    return o;
}

// Grid detection's per-(sequence, cell) arrays behind the step's workspace: thresholds, candidate counts, quotas and
// selected counts, B * G words each.
struct GridWs {
    size_t thr, seg_count, quota, n_sel, total;
};

GridWs grid_ws(size_t base, int batch, int cells)
{
    GridWs g;
    const size_t words = (size_t)batch * cells * 4;
    g.thr = align_up(base, 256);
    g.seg_count = align_up(g.thr + words, 256);
    g.quota = align_up(g.seg_count + words, 256);
    g.n_sel = align_up(g.quota + words, 256);
    g.total = align_up(g.n_sel + words, 256);
    return g;
}

// Grows the pinned landing zone of klt_frame_step_batch (every call has synchronised before it returned).
klt_status ensure_step_host(klt_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_step_bytes) return KLT_OK;
    return grow_ws(ctx, ctx->h_step, ctx->h_step_bytes, bytes, 1 << 16,
                   [](uint8_t** p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocDefault); }, cudaFreeHost);
}

// The whole step for the batch, enqueued on `st` without a synchronisation, an allocation or a host-side copy (a CUDA
// graph can hold it).  Arguments as klt_frame_step_batch_async, except: d_flags null = the workspace's flag word (cleared
// by the step), and out_stride must be at least min_out_stride.  out_stride caps each sequence's survivors + new corners.
// d_init (may be null): the forward pass's in/out start positions (klt_frame_step_batch_init_async).  reverse: the second
// pass runs from the new frame back into the old one (klt_frame_step_batch_fb_async), and d_bidir_err (may be null)
// receives each input slot's error.  grid_cols > 0: grid detection (klt_frame_step_batch_grid_async) on a grid_cols x
// grid_rows grid with tracks_per_cell, in a workspace of klt_frame_step_grid_ws_bytes.
klt_status frame_step_enqueue(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr, const uint8_t* d_next_img,
                              const uint8_t* d_next_pyr, const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride,
                              int n_seqs, const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                              float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                              int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                              int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                              int64_t min_out_stride, void* d_ws, int64_t ws_bytes, const klt_step_control* ctl, float* d_init,
                              bool reverse, float* d_bidir_err, double min_track_distance, uint8_t* d_thinned, cudaStream_t st,
                              int grid_cols = 0, int grid_rows = 0, int tracks_per_cell = 0)
{
    if (!ctx || !params || !d_prev_img || !d_next_img || !d_counts || !d_out_pts || !d_next_counts || !d_n_new || !d_ws)
        return KLT_ERR_INVALID_ARG;
    if (n_seqs < 1 || n_per_seq < 0 || (n_per_seq > 0 && (!d_pts || !d_keep))) return KLT_ERR_INVALID_ARG;
    const bool ids = d_ids_out != nullptr;
    if (ids != (d_next_id != nullptr) || (ids && n_per_seq > 0 && !d_ids_in) || (!ids && d_ids_in)) return KLT_ERR_INVALID_ARG;
    if (ctl && (!ctl->d_restarted || (ctl->d_restart && (!ctl->d_restart_pts || !ctl->d_restart_counts ||
                                                          ids != (ctl->d_restart_ids != nullptr) || ids != (ctl->d_restart_next_id != nullptr)))))
        return KLT_ERR_INVALID_ARG;
    klt_status s = check_layout(layout);
    if (s != KLT_OK) return s;
    if (pair_stride < 1 || prev_first < 0 || next_first < 0 ||
        (int64_t)prev_first + (int64_t)(n_seqs - 1) * pair_stride >= layout->batch ||
        (int64_t)next_first + (int64_t)(n_seqs - 1) * pair_stride >= layout->batch)
        return KLT_ERR_INVALID_ARG;
    if (layout->top > 0 && (!d_prev_pyr || !d_next_pyr)) return KLT_ERR_INVALID_ARG;
    if (params->win_w <= 2 || params->win_h <= 2 || (params->flags & KLT_OPTFLOW_USE_INITIAL_FLOW)) return KLT_ERR_INVALID_ARG;
    // goodFeaturesToTrack's assertions, then this entry point's own limits: maxCorners = 0 (no limit in cv2) would leave the
    // output width unbounded
    if (!(quality_level > 0) || !(min_distance >= 0) || max_corners < 0 || block_size < 1 || mask_radius < 0) return KLT_ERR_INVALID_ARG;
    if (max_corners == 0 || mask_radius > 127) return KLT_ERR_UNSUPPORTED;
    if (out_stride < min_out_stride || out_stride < n_per_seq || out_stride > 0x7fffffff) return KLT_ERR_INVALID_ARG;
    const klt_level& l0 = layout->level[0];
    const int w = l0.w, h = l0.h;
    if (block_size / 2 >= w || block_size / 2 >= h || w > 65535 || h > 65535 || n_seqs > 21845) return KLT_ERR_UNSUPPORTED;
    const StepWs o = step_ws(w, h, n_seqs, n_per_seq);
    const bool grid = grid_cols > 0;
    if (grid && (grid_cols > w || grid_rows < 1 || grid_rows > h || tracks_per_cell < 1)) return KLT_ERR_INVALID_ARG;
    if (grid && (int64_t)grid_cols * grid_rows > KLT_MAX_GRID_CELLS) return KLT_ERR_UNSUPPORTED;
    const GridWs g = grid_ws(o.total, n_seqs, grid ? grid_cols * grid_rows : 0);
    if (ws_bytes < (int64_t)(grid ? g.total : o.total) || ((uintptr_t)d_ws & 255)) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    uint8_t* d = static_cast<uint8_t*>(d_ws);
    int* d_surv = reinterpret_cast<int*>(d + o.surv);
    unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(d + o.keys);
    const long long px = (long long)w * h;
    if (!d_flags) d_flags = reinterpret_cast<uint32_t*>(d + o.flag);
    KLT_CUDA(cudaMemsetAsync(d + o.flag, 0, o.zero_end - o.flag, st));

    // 1. forward pass and the reference's second pass (same pair, started from the forward result), per-sequence counts.
    // With start positions, the forward pass reads them from d_init (cv2's OPTFLOW_USE_INITIAL_FLOW) and writes its result
    // there; the second pass starts from that result as always.
    // reverse: the second pass tracks p1 from the new frame back into the old one (the views swapped, the same launch
    // shape).  With start positions it starts at the mirrored start b = p1 - (s - p0): s is copied into p0r's region
    // before the forward pass overwrites d_init, and turned into b in place after it.
    float* d_p1 = d_init ? d_init : reinterpret_cast<float*>(d + o.p1);
    float* d_p0r = reinterpret_cast<float*>(d + o.p0r);
    if (n_per_seq > 0) {
        const bool mirror = reverse && d_init;
        if (mirror) KLT_CUDA(cudaMemcpyAsync(d_p0r, d_init, (size_t)n_seqs * n_per_seq * 8, cudaMemcpyDeviceToDevice, st));
        LKLaunch L;
        make_view(layout, d_prev_img, d_prev_pyr, prev_first, pair_stride, L.prev);
        make_view(layout, d_next_img, d_next_pyr, next_first, pair_stride, L.next);
        L.prev_pts = d_pts; L.next_pts = d_p1; L.status = d + o.status; L.err = reinterpret_cast<float*>(d + o.err); L.iters = nullptr;
        L.n_per_pair = n_per_seq;
        L.batch = n_seqs;
        L.counts = d_counts;
        set_lk_params(L, params);
        if (d_init) L.flags |= KLT_OPTFLOW_USE_INITIAL_FLOW;
        s = lk_launch(L, ctx->sm_count, st);
        if (s != KLT_OK) return s;
        if (mirror) {
            s = track_mirror_start_launch(d_pts, d_p1, d_counts, n_seqs, n_per_seq, d_p0r, st);
            if (s != KLT_OK) return s;
        }
        if (reverse) std::swap(L.prev, L.next);
        L.prev_pts = d_p1; L.next_pts = d_p0r; L.flags = params->flags | (mirror ? KLT_OPTFLOW_USE_INITIAL_FLOW : 0);
        s = lk_launch(L, ctx->sm_count, st);
        if (s != KLT_OK) return s;
    }
    // 2. filter, survivors (and their ids) compacted to the front of each output row.  min_track_distance > 0: the
    // compaction also thins the survivors; its grid's cell heads go in the eigenvalue map and its links in LK's err
    // region, both free until step 4
    TrackThin thin{min_track_distance, d_thinned, reinterpret_cast<int*>(d + o.eig), px, reinterpret_cast<unsigned*>(d + o.err)};
    s = track_compact_launch(d_pts, d_p1, d_p0r, d_counts, n_seqs, n_per_seq, max_bidir_error, w, h, d_keep, d_out_pts, out_stride,
                             d_surv, d_flags, n_per_seq > 0 ? d_ids_in : nullptr, n_per_seq > 0 ? d_ids_out : nullptr, ctl, d_next_id,
                             d_bidir_err, min_track_distance > 0 ? &thin : nullptr, st);
    if (s != KLT_OK) return s;
    // 3. detection mask around the survivors; 4. eigenvalues, candidates, key sorts; 5. greedy selection behind the survivors
    uint8_t* d_mask = d + o.mask;
    s = corner_mask_from_points_launch(d_out_pts, out_stride, d_surv, n_per_seq, n_seqs, mask_radius, w, h, d_mask, w, px, st);
    if (s != KLT_OK) return s;
    float* d_eig = reinterpret_cast<float*>(d + o.eig);
    if (grid) {
        // 4. eigenvalues; per-cell quotas from the survivors; per cell: threshold, candidates, sorts and selection (bitmaps
        // of cells too large for shared memory in the eigenvalue map, as below); 5. the cells' corners interleaved by rank
        int* d_quota = reinterpret_cast<int*>(d + g.quota);
        int* d_n_sel = reinterpret_cast<int*>(d + g.n_sel);
        s = corner_min_eig_launch(d_next_img + (int64_t)next_first * l0.batch_stride, l0.pitch, l0.batch_stride * pair_stride, w, h, n_seqs,
                                  block_size, d_eig, w, px, d_mask, w, px, nullptr, d + o.cws, st);
        if (s != KLT_OK) return s;
        s = corner_grid_quota_launch(d_out_pts, out_stride, d_surv, (int)out_stride, n_seqs, w, h, grid_cols, grid_rows, tracks_per_cell,
                                     d_quota, st);
        if (s != KLT_OK) return s;
        s = corner_grid_detect_launch(d_eig, w, px, w, h, n_seqs, d_mask, w, px, grid_cols, grid_rows, quality_level, min_distance, max_corners,
                                      out_stride, d_surv, d_quota, reinterpret_cast<float*>(d + g.thr), reinterpret_cast<unsigned*>(d + g.seg_count),
                                      d_n_sel, d_keys, px, reinterpret_cast<unsigned long long*>(d + o.cws), px, reinterpret_cast<unsigned*>(d_eig),
                                      px, st);
        if (s != KLT_OK) return s;
        return corner_grid_interleave_launch(d_keys, px, d_n_sel, w, h, n_seqs, grid_cols, grid_rows, max_corners, out_stride, d_surv, d_out_pts,
                                             out_stride, d_next_counts, d_n_new, d_ids_out, d_next_id, st);
    }
    unsigned* d_max = reinterpret_cast<unsigned*>(d + o.max);
    unsigned* d_count = reinterpret_cast<unsigned*>(d + o.count);
    s = corner_min_eig_launch(d_next_img + (int64_t)next_first * l0.batch_stride, l0.pitch, l0.batch_stride * pair_stride, w, h, n_seqs,
                              block_size, d_eig, w, px, d_mask, w, px, d_max, d + o.cws, st);
    if (s != KLT_OK) return s;
    s = corner_candidates_launch(d_eig, w, px, w, h, n_seqs, d_mask, w, px, d_max, quality_level, d_keys, px, (int)std::min<long long>(px, 0x7fffffff),
                                 d_count, st);
    if (s != KLT_OK) return s;
    unsigned long long* d_sorted = reinterpret_cast<unsigned long long*>(d + o.sorted);
    s = corner_sort_launch(d_keys, px, d_count, n_seqs, reinterpret_cast<unsigned*>(d + o.rank), d_sorted, 1 + kStepSortCap, kStepSortCap, st);
    if (s != KLT_OK) return s;
    s = corner_radix_sort_launch(d_keys, px, d_count, n_seqs, reinterpret_cast<unsigned long long*>(d + o.cws), px, st);
    if (s != KLT_OK) return s;
    return corner_select_launch(d_sorted, 1 + kStepSortCap, d_keys, px, w, h, n_seqs, min_distance, max_corners, out_stride, d_surv,
                                d_out_pts, out_stride, d_next_counts, d_n_new, d_ids_out, d_next_id, reinterpret_cast<unsigned*>(d_eig), px,
                                st);
}

}  // namespace

extern "C" {

int64_t klt_frame_step_ws_bytes(int w, int h, int batch, int n_per_seq)
{
    if (w < 1 || h < 1 || batch < 1 || n_per_seq < 0) return 0;
    return (int64_t)step_ws(w, h, batch, n_per_seq).total;
}

klt_status klt_frame_step_batch(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                int prev_first, int next_first, int pair_stride, int n_seqs,
                                const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                                int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                                int32_t* d_n_new, int32_t* next_counts, void* d_ws, int64_t ws_bytes, void* stream)
{
    if (!ctx || !next_counts) return KLT_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> step_lock(ctx->step_mutex);
    klt_status s = frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride,
                                      n_seqs, d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level,
                                      min_distance, block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, nullptr, nullptr,
                                      nullptr, nullptr, (int64_t)n_per_seq + max_corners, d_ws, ws_bytes, nullptr, nullptr, false, nullptr, 0.0, nullptr, st);
    if (s != KLT_OK) return s;
    // the one synchronisation: next counts and the bad-count flag (in the workspace) down
    KLT_DEVICE_GUARD(ctx);
    const size_t B = (size_t)n_seqs;
    s = ensure_step_host(ctx, B * 4 + 4);
    if (s != KLT_OK) return s;
    const uint8_t* d_flag = static_cast<const uint8_t*>(d_ws) + step_ws(layout->level[0].w, layout->level[0].h, n_seqs, n_per_seq).flag;
    KLT_CUDA(cudaMemcpyAsync(ctx->h_step, d_next_counts, B * 4, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaMemcpyAsync(ctx->h_step + B * 4, d_flag, 4, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    unsigned bad = 0;
    std::memcpy(&bad, ctx->h_step + B * 4, 4);
    if (bad) return KLT_ERR_INVALID_ARG;   // a count outside [0, n_per_seq]
    std::memcpy(next_counts, ctx->h_step, B * 4);
    return KLT_OK;
}

klt_status klt_frame_step_batch_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                      const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                      int prev_first, int next_first, int pair_stride, int n_seqs,
                                      const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                      float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                      double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                      int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                      int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes, void* stream)
{
    if (!d_flags) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, nullptr, nullptr, false, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}

klt_status klt_frame_step_batch_control_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                              const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                              int prev_first, int next_first, int pair_stride, int n_seqs,
                                              const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                              float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                              double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                              int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                              int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes,
                                              const klt_step_control* control, void* stream)
{
    if (!d_flags || !control) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, control, nullptr, false, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}

klt_status klt_frame_step_batch_init_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                           const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                           int prev_first, int next_first, int pair_stride, int n_seqs,
                                           const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                           float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                           double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                           int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                           int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes, float* d_init_pts,
                                           const klt_step_control* control, void* stream)
{
    if (!d_flags || (n_per_seq > 0 && !d_init_pts)) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, control, d_init_pts, false, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}

klt_status klt_frame_step_batch_fb_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                         const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                         int prev_first, int next_first, int pair_stride, int n_seqs,
                                         const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                         float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                         double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                         int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                         int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes, float* d_init_pts,
                                         const klt_step_control* control, float* d_bidir_err, void* stream)
{
    if (!d_flags) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, control, d_init_pts, true, d_bidir_err, 0.0, nullptr, (cudaStream_t)stream);
}

klt_status klt_frame_step_batch_thin_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                           const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                           int prev_first, int next_first, int pair_stride, int n_seqs,
                                           const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                           float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                           double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                           int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                           int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes, float* d_init_pts,
                                           const klt_step_control* control, float* d_bidir_err, int reverse,
                                           double min_track_distance, uint8_t* d_thinned, void* stream)
{
    // NaN fails both comparisons
    if (!(min_track_distance > 0.0) || std::isinf(min_track_distance)) return KLT_ERR_INVALID_ARG;
    if (min_track_distance > KLT_MAX_TRACK_DISTANCE) return KLT_ERR_UNSUPPORTED;
    if (!d_flags || (reverse != 0 && reverse != 1)) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, control, d_init_pts, reverse == 1, d_bidir_err, min_track_distance, d_thinned,
                              (cudaStream_t)stream);
}

int64_t klt_frame_step_grid_ws_bytes(int w, int h, int n_seqs, int n_per_seq, int cols, int rows)
{
    if (w < 1 || h < 1 || n_seqs < 1 || n_per_seq < 0 || cols < 1 || rows < 1 || (int64_t)cols * rows > KLT_MAX_GRID_CELLS) return 0;
    return (int64_t)grid_ws(step_ws(w, h, n_seqs, n_per_seq).total, n_seqs, cols * rows).total;
}

klt_status klt_frame_step_batch_grid_async(klt_ctx* ctx, const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                                           const uint8_t* d_next_img, const uint8_t* d_next_pyr, const klt_pyr_layout* layout,
                                           int prev_first, int next_first, int pair_stride, int n_seqs,
                                           const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                                           float max_bidir_error, int mask_radius, int max_corners, double quality_level,
                                           double min_distance, int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep,
                                           int32_t* d_next_counts, int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out,
                                           int32_t* d_next_id, uint32_t* d_flags, void* d_ws, int64_t ws_bytes, float* d_init_pts,
                                           const klt_step_control* control, float* d_bidir_err, int reverse,
                                           double min_track_distance, uint8_t* d_thinned, int cols, int rows, int tracks_per_cell,
                                           void* stream)
{
    // min_track_distance 0: no thinning; otherwise as klt_frame_step_batch_thin_async (NaN fails both comparisons)
    if (min_track_distance != 0.0 && (!(min_track_distance > 0.0) || std::isinf(min_track_distance))) return KLT_ERR_INVALID_ARG;
    if (min_track_distance > KLT_MAX_TRACK_DISTANCE) return KLT_ERR_UNSUPPORTED;
    if (cols < 1 || rows < 1 || tracks_per_cell < 1) return KLT_ERR_INVALID_ARG;
    if ((int64_t)cols * rows > KLT_MAX_GRID_CELLS) return KLT_ERR_UNSUPPORTED;
    if (!d_flags || (reverse != 0 && reverse != 1)) return KLT_ERR_INVALID_ARG;
    return frame_step_enqueue(ctx, d_prev_img, d_prev_pyr, d_next_img, d_next_pyr, layout, prev_first, next_first, pair_stride, n_seqs,
                              d_pts, d_counts, n_per_seq, params, max_bidir_error, mask_radius, max_corners, quality_level, min_distance,
                              block_size, d_out_pts, out_stride, d_keep, d_next_counts, d_n_new, d_ids_in, d_ids_out, d_next_id, d_flags,
                              n_per_seq, d_ws, ws_bytes, control, d_init_pts, reverse == 1, d_bidir_err, min_track_distance, d_thinned,
                              (cudaStream_t)stream, cols, rows, tracks_per_cell);
}

klt_status klt_track_records_step(klt_ctx* ctx, int n_seqs, int n_per_seq, int64_t out_stride, const uint8_t* d_keep,
                                  const float* d_out_pts, const int32_t* d_ids_out, const int32_t* d_next_counts,
                                  const float* d_first_pts_in, const int32_t* d_first_frames_in, float* d_first_pts_out,
                                  int32_t* d_first_frames_out, int32_t* d_frame, int depth, float* d_ring_pts, int32_t* d_ring_ids,
                                  int32_t* d_ring_src, int32_t* d_ring_counts, int32_t* d_ring_frames, void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return track_records_launch(d_keep, n_seqs, n_per_seq, d_out_pts, d_ids_out, out_stride, d_next_counts, d_first_pts_in, d_first_frames_in,
                                d_first_pts_out, d_first_frames_out, d_frame, depth, d_ring_pts, d_ring_ids, d_ring_src, d_ring_counts,
                                d_ring_frames, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

klt_status klt_track_records_step_control(klt_ctx* ctx, int n_seqs, int n_per_seq, int64_t out_stride, const uint8_t* d_keep,
                                          const float* d_out_pts, const int32_t* d_ids_out, const int32_t* d_next_counts,
                                          const float* d_first_pts_in, const int32_t* d_first_frames_in, float* d_first_pts_out,
                                          int32_t* d_first_frames_out, int32_t* d_frame, int depth, float* d_ring_pts, int32_t* d_ring_ids,
                                          int32_t* d_ring_src, int32_t* d_ring_counts, int32_t* d_ring_frames, const uint8_t* d_restarted,
                                          const int32_t* d_restart_counts, const float* d_restart_first_pts,
                                          const int32_t* d_restart_first_frames, void* stream)
{
    if (!ctx || !d_restarted || !d_restart_counts) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return track_records_launch(d_keep, n_seqs, n_per_seq, d_out_pts, d_ids_out, out_stride, d_next_counts, d_first_pts_in, d_first_frames_in,
                                d_first_pts_out, d_first_frames_out, d_frame, depth, d_ring_pts, d_ring_ids, d_ring_src, d_ring_counts,
                                d_ring_frames, d_restarted, d_restart_counts, d_restart_first_pts, d_restart_first_frames,
                                (cudaStream_t)stream);
}

klt_status klt_track_predict(klt_ctx* ctx, int n_seqs, int n_per_seq, const float* d_pts, const int32_t* d_counts,
                             const float* d_guess_pts, uint8_t* d_guess_mask, int depth, const float* d_ring_pts,
                             const int32_t* d_ring_src, const int32_t* d_ring_counts, const int32_t* d_frame, float* d_init_pts,
                             void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return track_predict_launch(d_pts, d_counts, n_seqs, n_per_seq, d_guess_pts, d_guess_mask, depth, d_ring_pts, d_ring_src, d_ring_counts,
                                d_frame, d_init_pts, (cudaStream_t)stream);
}

klt_status klt_track_window(klt_ctx* ctx, int n_seqs, int64_t width, int depth, const float* d_ring_pts, const int32_t* d_ring_src,
                            const int32_t* d_ring_counts, const int32_t* d_frame, int k, float* d_out, void* stream)
{
    if (!ctx) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return track_window_launch(d_ring_pts, d_ring_src, d_ring_counts, d_frame, depth, n_seqs, width, k, d_out, (cudaStream_t)stream);
}

// ---- bilateral pre-filter (SURVEY.md s8f rank 3; kernel in klt_bilateral.cu) -------------------------------------------

static klt_status bilateral_table(klt_ctx* ctx, int d, double sigma_color, double sigma_space, int* radius, int* n_taps, const float** d_tab)
{
    std::lock_guard<std::mutex> guard(ctx->cache_mutex);
    for (const auto& t : ctx->bilateral_tabs)
        if (t.d == d && t.sigma_color == sigma_color && t.sigma_space == sigma_space) {
            *radius = t.radius; *n_taps = t.n_taps; *d_tab = t.d_tab;
            return KLT_OK;
        }
    std::vector<float> tab;
    try { tab.resize((size_t)bilateral_table_capacity()); } catch (const std::bad_alloc&) { return KLT_ERR_OUT_OF_MEMORY; }
    const int n = bilateral_tables(d, sigma_color, sigma_space, tab.data(), (int)tab.size());
    if (n < 0) return KLT_ERR_UNSUPPORTED;
    if (ctx->bilateral_tabs.size() >= 64) return KLT_ERR_UNSUPPORTED;   // parameter sets are configuration, not data
    float* dev = nullptr;
    cudaError_t e = cudaMalloc(&dev, (size_t)(256 + 2 * n) * sizeof(float));
    if (e != cudaSuccess) return cuda_status(e);
    e = cudaMemcpy(dev, tab.data(), (size_t)(256 + 2 * n) * sizeof(float), cudaMemcpyHostToDevice);   // once per parameter set
    if (e == cudaSuccess) e = cudaDeviceSynchronize();   // (a pageable H2D copy may return before its DMA has landed)
    if (e != cudaSuccess) { cudaFree(dev); return (klt_status)e; }
    klt_ctx::BilateralTab t = {d, sigma_color, sigma_space, bilateral_radius(d, sigma_space), n, dev};
    try { ctx->bilateral_tabs.push_back(t); } catch (const std::bad_alloc&) { cudaFree(dev); return KLT_ERR_OUT_OF_MEMORY; }
    *radius = t.radius; *n_taps = n; *d_tab = dev;
    return KLT_OK;
}

klt_status klt_bilateral_filter(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_batch_stride,
                                uint8_t* d_dst, int64_t dst_pitch, int64_t dst_batch_stride, int batch, int d, double sigma_color,
                                double sigma_space, void* stream)
{
    if (!ctx || !d_src || !d_dst || w < 1 || h < 1 || batch < 1 || src_pitch < w || dst_pitch < w) return KLT_ERR_INVALID_ARG;
    if (d_src == d_dst) return KLT_ERR_INVALID_ARG;   // not an in-place filter (cv2 does not allow it either)
    KLT_DEVICE_GUARD(ctx);
    int radius = 0, n_taps = 0;
    const float* d_tab = nullptr;
    klt_status s = bilateral_table(ctx, d, sigma_color, sigma_space, &radius, &n_taps, &d_tab);
    if (s != KLT_OK) return s;
    return bilateral_launch(d_src, w, h, src_pitch, src_batch_stride, d_dst, dst_pitch, dst_batch_stride, batch, radius, n_taps, d_tab,
                            (cudaStream_t)stream);
}

klt_status klt_bilateral_filter_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, int d, double sigma_color,
                                     double sigma_space, uint8_t* out, int64_t out_pitch)
{
    if (!ctx || !img || !out || w < 1 || h < 1 || pitch < w || out_pitch < w) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    int radius = 0, n_taps = 0;
    const float* d_tab = nullptr;
    klt_status s = bilateral_table(ctx, d, sigma_color, sigma_space, &radius, &n_taps, &d_tab);
    if (s != KLT_OK) return s;
    const size_t img_bytes = upload_bytes(pitch, w, h);
    const size_t opitch = align_up((size_t)w, 128);
    const size_t out_bytes = opitch * (size_t)h;
    s = claim_device_ws(ctx, img_bytes + out_bytes, nullptr, nullptr);
    if (s != KLT_OK) return s;
    s = ensure_host_ws(ctx, out_bytes);
    if (s != KLT_OK) return s;
    uint8_t* dws = ctx->d_ws;
    cudaStream_t st = ctx->stream;
    // Pageable input (what cv2.imread returns): staged through the pinned landing zone by the calling thread and the
    // helper threads, like the images of the tracking entry point.  The result lands in the pinned staging buffer with
    // one contiguous DMA and is copied out row by row by the CPU (a D2H copy into pageable memory is staged by the
    // driver, synchronously and slowly).
    const size_t raw = raw_span(pitch, w, h);
    const uint8_t* src = img;
    if (near_contiguous(raw, w, h) && raw >= (128u << 10) && is_pageable(img)) {
        s = ensure_host_in(ctx, align_up(raw, 256));
        if (s != KLT_OK) return s;
        const uint8_t* none = nullptr;
        if (klt_ctx::Stager* stager = stage_pageable(ctx, src, raw, none, 0, 0)) {
            stager->finish_job(0);
            stager->finish_job(1);
        }
    }
    int64_t dpitch = 0;
    s = upload_u8(dws, &dpitch, src, pitch, w, h, st);
    if (s != KLT_OK) return s;
    s = bilateral_launch(dws, w, h, dpitch, 0, dws + img_bytes, (long long)opitch, 0, 1, radius, n_taps, d_tab, st);
    if (s != KLT_OK) return s;
    KLT_CUDA(cudaMemcpyAsync(ctx->h_ws, dws + img_bytes, out_bytes, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    if ((size_t)out_pitch == (size_t)w && opitch == (size_t)w) {
        std::memcpy(out, ctx->h_ws, out_bytes);
    } else {
        for (int y = 0; y < h; ++y) std::memcpy(out + (size_t)y * (size_t)out_pitch, ctx->h_ws + (size_t)y * opitch, (size_t)w);
    }
    return KLT_OK;
}

// ---- sub-pixel corner refinement (kernel in klt_subpix.cu) ----------------------------------------------------------------

static klt_status subpix_check(int w, int h, int64_t pitch, int batch, int win_w, int win_h)
{
    if (batch < 1 || win_w < 1 || win_h < 1 || w < 2 * win_w + 5 || h < 2 * win_h + 5 || pitch < w) return KLT_ERR_INVALID_ARG;
    if (win_w > KLT_MAX_SUBPIX_WIN || win_h > KLT_MAX_SUBPIX_WIN || batch > 65535) return KLT_ERR_UNSUPPORTED;
    return KLT_OK;
}

klt_status klt_corner_sub_pix(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride, int batch,
                              float* d_pts, int64_t row_stride, const int32_t* d_end, const int32_t* d_n, int win_w, int win_h,
                              int zero_w, int zero_h, int crit_type, int max_count, double eps, void* stream)
{
    if (!ctx || !d_img || !d_pts || !d_end || !d_n || row_stride < 0) return KLT_ERR_INVALID_ARG;
    klt_status s = subpix_check(w, h, pitch, batch, win_w, win_h);
    if (s != KLT_OK) return s;
    KLT_DEVICE_GUARD(ctx);
    return subpix_launch(d_img, w, h, pitch, batch_stride, batch, d_pts, row_stride, d_end, d_n, win_w, win_h, zero_w, zero_h,
                         crit_type, max_count, eps, (cudaStream_t)stream);
}

klt_status klt_corner_sub_pix_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, float* pts, int n, int win_w,
                                   int win_h, int zero_w, int zero_h, int crit_type, int max_count, double eps)
{
    if (!ctx || !img || n < 0 || (n > 0 && !pts)) return KLT_ERR_INVALID_ARG;
    klt_status s = subpix_check(w, h, pitch, 1, win_w, win_h);
    if (s != KLT_OK) return s;
    if (n == 0) return KLT_OK;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    const size_t img_bytes = upload_bytes(pitch, w, h);
    const size_t pts_bytes = align_up((size_t)n * 2 * sizeof(float), 256);
    s = claim_device_ws(ctx, img_bytes + pts_bytes + 256, nullptr, nullptr);
    if (s != KLT_OK) return s;
    s = ensure_host_ws(ctx, pts_bytes + 256);
    if (s != KLT_OK) return s;
    uint8_t* dws = ctx->d_ws;
    float* d_pts = reinterpret_cast<float*>(dws + img_bytes);
    int32_t* d_cnt = reinterpret_cast<int32_t*>(dws + img_bytes + pts_bytes);
    cudaStream_t st = ctx->stream;
    // the points and the count go up through the pinned staging buffer (one DMA), the image like the other host calls
    std::memcpy(ctx->h_ws, pts, (size_t)n * 2 * sizeof(float));
    std::memcpy(ctx->h_ws + pts_bytes, &n, sizeof(int32_t));
    int64_t dpitch = 0;
    s = upload_u8(dws, &dpitch, img, pitch, w, h, st);
    if (s != KLT_OK) return s;
    KLT_CUDA(cudaMemcpyAsync(d_pts, ctx->h_ws, pts_bytes + sizeof(int32_t), cudaMemcpyHostToDevice, st));
    s = subpix_launch(dws, w, h, dpitch, 0, 1, d_pts, n, d_cnt, d_cnt, win_w, win_h, zero_w, zero_h, crit_type, max_count, eps, st);
    if (s != KLT_OK) return s;
    KLT_CUDA(cudaMemcpyAsync(ctx->h_ws, d_pts, (size_t)n * 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    std::memcpy(pts, ctx->h_ws, (size_t)n * 2 * sizeof(float));
    return KLT_OK;
}

// ---- contrast-limited histogram equalisation (kernels in klt_clahe.cu) ---------------------------------------------------

int64_t klt_clahe_ws_bytes(int batch, int tiles_x, int tiles_y)
{
    if (batch < 1 || tiles_x < 1 || tiles_y < 1) return 0;
    return (int64_t)clahe_lut_bytes(batch, tiles_x, tiles_y);
}

klt_status klt_clahe(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_batch_stride, uint8_t* d_dst,
                     int64_t dst_pitch, int64_t dst_batch_stride, int batch, double clip_limit, int tiles_x, int tiles_y, void* d_ws,
                     int64_t ws_bytes, void* stream)
{
    if (!ctx || !d_src || !d_dst || !d_ws || batch < 1 || src_pitch < w || dst_pitch < w) return KLT_ERR_INVALID_ARG;
    if (d_src == d_dst && (src_pitch != dst_pitch || (batch > 1 && src_batch_stride != dst_batch_stride))) return KLT_ERR_INVALID_ARG;
    ClahePlan plan;
    klt_status s = clahe_plan(w, h, clip_limit, tiles_x, tiles_y, &plan);
    if (s != KLT_OK) return s;
    if (batch > 65535) return KLT_ERR_UNSUPPORTED;
    if (ws_bytes < clahe_lut_bytes(batch, tiles_x, tiles_y)) return KLT_ERR_INVALID_ARG;
    KLT_DEVICE_GUARD(ctx);
    return clahe_launch(d_src, w, h, src_pitch, src_batch_stride, d_dst, dst_pitch, dst_batch_stride, batch, plan,
                        static_cast<uint8_t*>(d_ws), (cudaStream_t)stream);
}

klt_status klt_clahe_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, double clip_limit, int tiles_x, int tiles_y,
                          uint8_t* out, int64_t out_pitch)
{
    if (!ctx || !img || !out || pitch < w || out_pitch < w) return KLT_ERR_INVALID_ARG;
    ClahePlan plan;
    klt_status s = clahe_plan(w, h, clip_limit, tiles_x, tiles_y, &plan);
    if (s != KLT_OK) return s;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    const size_t img_bytes = upload_bytes(pitch, w, h);
    const size_t opitch = align_up((size_t)w, 128);
    const size_t out_bytes = opitch * (size_t)h;
    const size_t lut_off = img_bytes + align_up(out_bytes, 256);
    s = claim_device_ws(ctx, lut_off + (size_t)clahe_lut_bytes(1, tiles_x, tiles_y), nullptr, nullptr);
    if (s != KLT_OK) return s;
    s = ensure_host_ws(ctx, out_bytes);
    if (s != KLT_OK) return s;
    uint8_t* dws = ctx->d_ws;
    cudaStream_t st = ctx->stream;
    int64_t dpitch = 0;
    s = upload_u8(dws, &dpitch, img, pitch, w, h, st);
    if (s != KLT_OK) return s;
    s = clahe_launch(dws, w, h, dpitch, 0, dws + img_bytes, (long long)opitch, 0, 1, plan, dws + lut_off, st);
    if (s != KLT_OK) return s;
    KLT_CUDA(cudaMemcpyAsync(ctx->h_ws, dws + img_bytes, out_bytes, cudaMemcpyDeviceToHost, st));
    KLT_CUDA(cudaStreamSynchronize(st));
    if ((size_t)out_pitch == (size_t)w && opitch == (size_t)w) {
        std::memcpy(out, ctx->h_ws, out_bytes);
    } else {
        for (int y = 0; y < h; ++y) std::memcpy(out + (size_t)y * (size_t)out_pitch, ctx->h_ws + (size_t)y * opitch, (size_t)w);
    }
    return KLT_OK;
}

// Diagnostics (not part of include/klt_b200.h): number of pyramids the host entry points of this context did NOT rebuild
// because the uploaded image was unchanged.  Synchronises the context's stream.
int klt_debug_pyr_reuse_count(klt_ctx* ctx, unsigned long long* skipped)
{
    if (!ctx || !skipped) return KLT_ERR_INVALID_ARG;
    *skipped = 0;
    if (!ctx->d_hash) return KLT_OK;
    KLT_DEVICE_GUARD(ctx);
    std::lock_guard<std::mutex> host_lock(ctx->host_mutex);
    KLT_CUDA(cudaStreamSynchronize(ctx->stream));
    KLT_CUDA(cudaMemcpy(skipped, ctx->d_hash + 16, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return KLT_OK;
}

}  // extern "C"
