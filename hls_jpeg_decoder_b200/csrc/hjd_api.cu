// csrc/hjd_api.cu -- the C ABI of include/hjd.h: batch handle, HBM slabs, launches.
//
// Host-side counterpart of the reference's ConvertJpgFile / JpegDecodeHW call sequence
// (openjpg.cpp:593-684): load -> parse -> decode -> (write BMP).  Here "decode" is a set of
// kernel launches over flat HBM slabs holding N images, and nothing is decoded on the CPU.
// What an upload computes on the host is planned by csrc/batch_plan.cpp; this file sizes the slabs from the plan,
// copies it to the device and launches the kernels.
#include "../../include/hjd.h"
#include "hjd_types.h"
#include "jpeg_parse.h"
#include "batch_plan.h"
#include "kernels.cuh"
#include "selfsync.cuh"
#include "multiscan.cuh"
#include "scaled.cuh"
#include "orient.cuh"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <atomic>
#include <memory>
#include <string>
#include <vector>

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static_assert(HJD_MAX_SCANS == HJD_MAX_SCANS_PER_IMAGE, "hjd_types.h and include/hjd.h state the same scan cap");

static thread_local std::string g_err;

static int fail(int code, const char* what, const char* detail = nullptr)
{
    g_err = what;
    if (detail) { g_err += ": "; g_err += detail; }
    return code;
}

#define CU(call)                                                                     \
    do {                                                                             \
        cudaError_t e_ = (call);                                                     \
        if (e_ != cudaSuccess) return fail(HJD_ERR_CUDA, #call, cudaGetErrorString(e_)); \
    } while (0)

// ------------------------------------------------------------------------------------------
// grow-only buffers, freed with their owner
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = bytes + bytes / 16 + 4096;      // slack so that slowly growing batches do not reallocate
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&p, want); }
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(const PinBuf&) = delete;
    PinBuf& operator=(const PinBuf&) = delete;
    ~PinBuf() { if (p) cudaFreeHost(p); }
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

// ------------------------------------------------------------------------------------------
// batch
// ------------------------------------------------------------------------------------------
#define HJD_NSTREAMS 3

struct hjd_batch {
    int device = 0;
    unsigned flags = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t mark[HJD_MARK_SLOTS] = {};                          // hjd_batch_mark
    cudaStream_t aux[HJD_NSTREAMS] = {nullptr, nullptr, nullptr}; // chunk streams
    cudaEvent_t ev_fork = nullptr, ev_join[HJD_NSTREAMS] = {nullptr, nullptr, nullptr};
    std::vector<FileRef> files;
    const uint8_t* contig_src = nullptr;      // host address of device-arena offset 0 (arena uploads)
    uint64_t arena_bytes = 0;
    int overlap = 1;                                               // 0: one chunk, one stream (stage timings)
    int chunk_images = 0;                                          // > 0: images per chunk asked for by the caller of hjd_batch_decode_host
    uint32_t ss_range_req = 0;                  // 0 = automatic
    int max_sync_ctas = 1;                      // grid limit of the cooperative synchronisation kernel on this device
    int sm_count = 148;                         // multiprocessors of this device (work-list balancing)

    BatchPlan plan;                             // host state of the uploaded batch (reset by every upload)
    bool uploaded = false, decoded = false;

    // the last decode
    bool ss_ran = false;                        // it ran kernel 1b (its round count is in d_flag)
    int launches = 0;
    int tc_chunks = 0, cc_chunks = 0;           // chunks whose MCUs went through the tensor-core / CUDA-core fused kernel
    int sc_chunks = 0;                          // ... through the scaled kernel (HJD_FLAG_SCALE_*)
    int gy_chunks = 0;                          // ... through a luma-only kernel (HJD_FLAG_GRAY_OUT)

    DevBuf d_arena, d_imgs, d_tsets, d_qsets, d_work, d_segs, d_mcucta, d_lumacta, d_slices, d_slicecnt, d_istart, d_coef, d_planes, d_rgb, d_status;
    DevBuf d_scans, d_mswork, d_msstarts, d_mstabs;
    DevBuf d_ojobs, d_otiles;                   // HJD_FLAG_EXIF_ORIENT
    DevBuf d_ss, d_sswork, d_sssegs, d_destuff, d_dlen, d_counts, d_scantmp, d_ssE0, d_ssX, d_ssnb, d_flag;
    PinBuf h_meta, h_out;                       // h_out: staging of the single-image calls
};

// The reduced IDCT's cosine table for N samples per block side (host libm); N = 8 is the full IDCT's
// (loadjpg.cpp:96-102).
static void compute_scaled_cos(int n, float* cos_n)
{
    const float PI = 3.14f;
    for (int p = 0; p < n; p++)
        for (int k = 0; k < n; k++) cos_n[p * n + k] = cosf(((2 * p + 1) * k * PI) / (float)(2 * n));
}

static void compute_idct_constants(float cos_tab[64], float* cc0, float* cc00)
{
    // The very expressions of the reference, evaluated by the host libm (loadjpg.cpp:96-102,108,120).
    compute_scaled_cos(8, cos_tab);
    volatile float c0 = 1.0f / sqrtf(2);
    *cc0 = c0 * 1.0f;
    *cc00 = c0 * c0;
}

extern "C" void hjd_get_idct_tables(float cos_tab[64], float cc[64])
{
    float c0, c00;
    compute_idct_constants(cos_tab, &c0, &c00);
    for (int u = 0; u < 8; u++)
        for (int v = 0; v < 8; v++) cc[u * 8 + v] = (u == 0 && v == 0) ? c00 : ((u == 0 || v == 0) ? c0 : 1.0f);
}

extern "C" void hjd_get_idct_matrix(uint16_t img[8192])
{
    float cos_tab[64], c0, c00;
    compute_idct_constants(cos_tab, &c0, &c00);
    hjd_build_idct_matrix(cos_tab, c0, c00, img);
}

extern "C" int hjd_version(void) { return HJD_VERSION; }
extern "C" const char* hjd_last_error(void) { return g_err.c_str(); }

extern "C" int hjd_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" hjd_batch* hjd_batch_create(int device, unsigned flags)
{
    if ((flags & HJD_FLAG_EXIF_ORIENT) && (flags & HJD_FLAG_BMP_OUT)) {
        fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_EXIF_ORIENT does not combine with HJD_FLAG_BMP_OUT (the BMP layout is "
                                              "bottom-up with padded rows; the orientation pass writes top-down RGB24 or luma)");
        return nullptr;                  // checked first: it does not depend on the device
    }
    int n = hjd_device_count();
    if (n <= 0) { fail(HJD_ERR_CUDA, "hjd_batch_create", "no CUDA device available (this library has no CPU fallback)"); return nullptr; }
    if (device < 0 || device >= n) { fail(HJD_ERR_ARG, "hjd_batch_create", "bad device index"); return nullptr; }
    if ((flags & HJD_FLAG_BMP_OUT) && (flags & HJD_FLAG_KEEP_PLANES)) { fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_BMP_OUT is an epilogue of the default (fused) kernels"); return nullptr; }
    if ((flags & HJD_FLAG_SCALE_MASK) &&
        (flags & (HJD_FLAG_KEEP_PLANES | HJD_FLAG_BMP_OUT | HJD_FLAG_TENSOR_CORE_IDCT | HJD_FLAG_CUDA_CORE_IDCT))) {
        fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_SCALE_* has no planes, no BMP output and its own kernel: it combines with "
                                              "none of HJD_FLAG_KEEP_PLANES, HJD_FLAG_BMP_OUT, HJD_FLAG_TENSOR_CORE_IDCT, HJD_FLAG_CUDA_CORE_IDCT");
        return nullptr;
    }
    if ((flags & HJD_FLAG_GRAY_OUT) &&
        (flags & (HJD_FLAG_KEEP_PLANES | HJD_FLAG_BMP_OUT | HJD_FLAG_TENSOR_CORE_IDCT | HJD_FLAG_CUDA_CORE_IDCT))) {
        fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_GRAY_OUT writes Y alone with its own kernel: it combines with none of "
                                              "HJD_FLAG_KEEP_PLANES (the planes already hold Y), HJD_FLAG_BMP_OUT (no 8-bit BMP), "
                                              "HJD_FLAG_TENSOR_CORE_IDCT, HJD_FLAG_CUDA_CORE_IDCT (RGB kernels)");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) { fail(HJD_ERR_CUDA, "cudaSetDevice"); return nullptr; }
    hjd_batch* b = new hjd_batch();
    b->device = device;
    b->flags = flags;
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    b->own_stream = true;
    for (int i = 0; i < 5 && e == cudaSuccess; i++) e = cudaEventCreate(&b->ev[i]);
    for (int i = 0; i < HJD_MARK_SLOTS && e == cudaSuccess; i++) e = cudaEventCreate(&b->mark[i]);
    for (int i = 0; i < HJD_NSTREAMS && e == cudaSuccess; i++) e = cudaStreamCreateWithFlags(&b->aux[i], cudaStreamNonBlocking);
    for (int i = 0; i < HJD_NSTREAMS && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&b->ev_join[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = hjd_kernels_init_device();            // function attributes are per device
    if (e == cudaSuccess) e = hjd_selfsync_init_device(&b->max_sync_ctas);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&b->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) {
        float cos_tab[64], c0, c00;
        compute_idct_constants(cos_tab, &c0, &c00);
        e = hjd_set_idct_constants(cos_tab, c0, c00);
        if (e == cudaSuccess) {
            float cos4[16], cos2[4], cos1[1], cc[64], cc16[16];
            compute_scaled_cos(4, cos4);
            compute_scaled_cos(2, cos2);
            compute_scaled_cos(1, cos1);
            hjd_get_idct_tables(cos_tab, cc);
            for (int u = 0; u < 4; u++)
                for (int v = 0; v < 4; v++) cc16[u * 4 + v] = cc[u * 8 + v];
            e = hjd_set_scaled_constants(cos4, cos2, cos1, cc16);
        }
    }
    if (e != cudaSuccess) {
        fail(HJD_ERR_CUDA, "hjd_batch_create", cudaGetErrorString(e));
        hjd_batch_destroy(b);
        return nullptr;
    }
    return b;
}

extern "C" void hjd_batch_destroy(hjd_batch* b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    for (int i = 0; i < 5; i++) if (b->ev[i]) cudaEventDestroy(b->ev[i]);
    for (int i = 0; i < HJD_MARK_SLOTS; i++) if (b->mark[i]) cudaEventDestroy(b->mark[i]);
    for (int i = 0; i < HJD_NSTREAMS; i++) { if (b->aux[i]) { cudaStreamSynchronize(b->aux[i]); cudaStreamDestroy(b->aux[i]); } if (b->ev_join[i]) cudaEventDestroy(b->ev_join[i]); }
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
    delete b;                                   // frees the slabs and the pinned buffers
}

extern "C" int hjd_batch_set_stream(hjd_batch* b, void* cuda_stream)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_stream", "null batch");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
    b->stream = (cudaStream_t)cuda_stream;
    b->own_stream = false;
    return HJD_OK;
}

// Device slabs of the planned batch.  They only grow, so a batch no larger than an earlier one allocates nothing.
static int ensure_slabs(hjd_batch* b)
{
    const BatchPlan& p = b->plan;
    const size_t n = p.imgs.size();
    CU(b->d_arena.ensure(b->arena_bytes + 64));
    CU(b->d_imgs.ensure(sizeof(HjdImageDesc) * (n + 1)));
    CU(b->d_tsets.ensure(sizeof(HjdTableSet) * (p.tsets.size() + 1)));
    CU(b->d_qsets.ensure(sizeof(HjdQuantSet) * (p.qsets.size() + 1)));
    CU(b->d_work.ensure(sizeof(HjdEntropyWork) * (p.work.size() + 1)));
    CU(b->d_segs.ensure(sizeof(HjdEntropySeg) * (p.segs.size() + 1)));
    CU(b->d_slices.ensure(sizeof(HjdScanSlice) * (p.slices.size() + 1)));
    CU(b->d_slicecnt.ensure(sizeof(uint32_t) * (p.slices.size() + 1)));
    CU(b->d_mcucta.ensure(sizeof(uint32_t) * (n + 2)));
    if (b->flags & HJD_FLAG_GRAY_OUT) CU(b->d_lumacta.ensure(sizeof(uint32_t) * (n + 2)));
    CU(b->d_istart.ensure(sizeof(uint32_t) * ((size_t)p.total_intervals + 2)));
    CU(b->d_coef.ensure(p.total_blocks * 128 + 256));
    CU(b->d_rgb.ensure(p.rgb_bytes + p.stage_bytes + 256));      // staging regions of oriented images behind the slab
    CU(b->d_status.ensure(sizeof(int32_t) * (n + 1)));
    if (b->flags & HJD_FLAG_KEEP_PLANES) CU(b->d_planes.ensure(p.plane_bytes + 256));
    if (!p.ss.empty()) {
        CU(b->d_ss.ensure(sizeof(HjdSsImage) * p.ss.size()));
        CU(b->d_sswork.ensure(sizeof(HjdSsWork) * p.sswork.size()));
        CU(b->d_sssegs.ensure(sizeof(HjdSsSeg) * (p.sssegs.size() + 1)));
        CU(b->d_destuff.ensure(p.ss_dst_bytes + 256));
        CU(b->d_dlen.ensure(sizeof(uint32_t) * p.ss.size()));
        CU(b->d_counts.ensure(sizeof(uint32_t) * ((size_t)p.ss_chunks + 2)));
        CU(b->d_scantmp.ensure(sizeof(uint32_t) * (size_t)p.ss_tmp_stride * (p.chunks.size() + 1)));
        CU(b->d_ssE0.ensure(sizeof(uint64_t) * (size_t)p.ss_subs));
        CU(b->d_ssX.ensure(sizeof(uint64_t) * (size_t)p.ss_subs));
        CU(b->d_ssnb.ensure(sizeof(uint32_t) * (4 * (size_t)p.ss_subs + 4)));
        CU(b->d_flag.ensure(sizeof(uint32_t) * 4 * (p.chunks.size() + 1)));
    }
    if (!p.scans.empty()) {
        CU(b->d_scans.ensure(sizeof(HjdScanDesc) * p.scans.size()));
        CU(b->d_mswork.ensure(sizeof(HjdMsWork) * p.mswork.size() + 16));
        CU(b->d_msstarts.ensure(sizeof(uint32_t) * p.ms_starts.size() + 16));
        CU(b->d_mstabs.ensure(sizeof(HjdHuffTable) * p.ms_tabs.size() + 16));
    }
    if (!p.orient_jobs.empty()) {
        CU(b->d_ojobs.ensure(sizeof(HjdOrientJob) * p.orient_jobs.size()));
        CU(b->d_otiles.ensure(sizeof(uint32_t) * p.orient_tiles.size()));
    }
    return HJD_OK;
}

// The plan's descriptor arrays to their slabs: packed at 256-byte offsets into one pinned block, one asynchronous
// copy each, and the status slab cleared.
static int stage_plan(hjd_batch* b)
{
    const BatchPlan& p = b->plan;
    struct Stage { DevBuf* dst; const void* src; size_t bytes; };
    const Stage stages[] = {
        {&b->d_imgs, p.imgs.data(), sizeof(HjdImageDesc) * p.imgs.size()},
        {&b->d_tsets, p.tsets.data(), sizeof(HjdTableSet) * p.tsets.size()},
        {&b->d_qsets, p.qsets.data(), sizeof(HjdQuantSet) * p.qsets.size()},
        {&b->d_work, p.work.data(), sizeof(HjdEntropyWork) * p.work.size()},
        {&b->d_istart, p.host_istart.data(), sizeof(uint32_t) * p.host_istart.size()},
        {&b->d_ss, p.ss.data(), sizeof(HjdSsImage) * p.ss.size()},
        {&b->d_sswork, p.sswork.data(), sizeof(HjdSsWork) * p.sswork.size()},
        {&b->d_segs, p.segs.data(), sizeof(HjdEntropySeg) * p.segs.size()},
        {&b->d_sssegs, p.sssegs.data(), sizeof(HjdSsSeg) * p.sssegs.size()},
        {&b->d_mcucta, p.mcu_cta.data(), sizeof(uint32_t) * p.mcu_cta.size()},
        {&b->d_lumacta, p.luma_cta.data(), sizeof(uint32_t) * p.luma_cta.size()},
        {&b->d_slices, p.slices.data(), sizeof(HjdScanSlice) * p.slices.size()},
        {&b->d_scans, p.scans.data(), sizeof(HjdScanDesc) * p.scans.size()},
        {&b->d_mswork, p.mswork.data(), sizeof(HjdMsWork) * p.mswork.size()},
        {&b->d_msstarts, p.ms_starts.data(), sizeof(uint32_t) * p.ms_starts.size()},
        {&b->d_mstabs, p.ms_tabs.data(), sizeof(HjdHuffTable) * p.ms_tabs.size()},
        {&b->d_ojobs, p.orient_jobs.data(), sizeof(HjdOrientJob) * p.orient_jobs.size()},
        {&b->d_otiles, p.orient_tiles.data(), p.orient_jobs.empty() ? 0 : sizeof(uint32_t) * p.orient_tiles.size()},
    };
    size_t total = 0;
    for (const Stage& s : stages) total = align_up(total, 256) + s.bytes;
    CU(b->h_meta.ensure(total + 256));
    uint8_t* hm = (uint8_t*)b->h_meta.p;
    size_t off = 0;
    for (const Stage& s : stages) {
        off = align_up(off, 256);
        if (s.bytes) {
            memcpy(hm + off, s.src, s.bytes);
            CU(cudaMemcpyAsync(s.dst->p, hm + off, s.bytes, cudaMemcpyHostToDevice, b->stream));
        }
        off += s.bytes;
    }
    CU(cudaMemsetAsync(b->d_status.p, 0, sizeof(int32_t) * (p.imgs.size() + 1), b->stream));
    return HJD_OK;
}

// Plan, slabs and descriptor copies of a batch.  b->files[i].dev_off must already hold the arena offset of
// file i.  The files themselves are copied by copy_files(), whole or chunk by chunk.
static int upload_common(hjd_batch* b, bool chunked)
{
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));     // staging buffers of the previous batch are free again
    b->plan = BatchPlan();
    b->uploaded = b->decoded = false;
    const PlanConfig cfg{b->flags, b->overlap, b->chunk_images, b->ss_range_req, b->sm_count, chunked};
    std::string err;
    if (hjd_plan_batch(b->files, cfg, &b->plan, &err) != HJD_OK) return fail(HJD_ERR_ARG, "hjd_batch_upload", err.c_str());
    int rc = ensure_slabs(b);
    if (rc == HJD_OK) rc = stage_plan(b);
    if (rc == HJD_OK) b->uploaded = true;
    return rc;
}

// Host -> device copy of the files of images [img0, img1) (one copy for arena uploads).
static int copy_files(hjd_batch* b, const Chunk& c, cudaStream_t st)
{
    if (c.arena_hi <= c.arena_lo) return HJD_OK;
    if (b->contig_src) {
        CU(cudaMemcpyAsync((uint8_t*)b->d_arena.p + c.arena_lo, b->contig_src + c.arena_lo, c.arena_hi - c.arena_lo,
                           cudaMemcpyHostToDevice, st));
    } else {
        for (int i = c.img0; i < c.img1; i++) {
            const FileRef& f = b->files[i];
            if (f.ptr && f.size > 0)
                CU(cudaMemcpyAsync((uint8_t*)b->d_arena.p + f.dev_off, f.ptr, (size_t)f.size, cudaMemcpyHostToDevice, st));
        }
    }
    return HJD_OK;
}

static int prepare_separate(hjd_batch* b, const uint8_t* const* bufs, const int64_t* sizes, int n, bool chunked)
{
    b->files.assign((size_t)n, FileRef{nullptr, 0, 0});
    uint64_t off = 0;
    for (int i = 0; i < n; i++) {
        b->files[i] = FileRef{bufs[i], sizes[i], off};
        off += align_up(sizes[i] > 0 ? (uint64_t)sizes[i] : 0, 16);
    }
    b->arena_bytes = off;
    b->contig_src = nullptr;
    return upload_common(b, chunked);
}

static int prepare_arena(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n,
                         bool chunked)
{
    b->files.assign((size_t)n, FileRef{nullptr, 0, 0});
    int64_t lo = n ? offsets[0] : 0, hi = 0;
    for (int i = 0; i < n; i++) {
        if (offsets[i] < 0 || sizes[i] < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "negative offset/size");
        if (i && offsets[i] < offsets[i - 1]) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "offsets must be ascending");
        if (offsets[i] < lo) lo = offsets[i];
        if (offsets[i] + sizes[i] > hi) hi = offsets[i] + sizes[i];
    }
    const int64_t lo_al = lo & ~(int64_t)15;      // keep the 16-byte phase of every file
    for (int i = 0; i < n; i++) b->files[i] = FileRef{arena + offsets[i], sizes[i], (uint64_t)(offsets[i] - lo_al)};
    b->arena_bytes = n ? (uint64_t)(hi - lo_al) : 0;
    b->contig_src = n ? arena + lo_al : nullptr;
    return upload_common(b, chunked);
}

extern "C" int hjd_batch_upload(hjd_batch* b, const uint8_t* const* bufs, const int64_t* sizes, int n)
{
    if (!b || !bufs || !sizes || n < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload", "bad arguments");
    int rc = prepare_separate(b, bufs, sizes, n, b->overlap > 1);
    if (rc) return rc;
    for (const Chunk& c : b->plan.chunks) { rc = copy_files(b, c, b->stream); if (rc) return rc; }
    return HJD_OK;
}

extern "C" int hjd_batch_upload_arena(hjd_batch* b, const uint8_t* arena, const int64_t* offsets,
                                      const int64_t* sizes, int n)
{
    if (!b || !arena || !offsets || !sizes || n < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "bad arguments");
    int rc = prepare_arena(b, arena, offsets, sizes, n, b->overlap > 1);
    if (rc) return rc;
    for (const Chunk& c : b->plan.chunks) { rc = copy_files(b, c, b->stream); if (rc) return rc; }
    return HJD_OK;
}

extern "C" int hjd_batch_set_overlap(hjd_batch* b, int on)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_overlap", "null batch");
    b->overlap = on < 0 ? 0 : on;     // 0 serial, 1 default chunking, > 1: target blocks per chunk; next upload
    return HJD_OK;
}

extern "C" int hjd_batch_set_selfsync_range(hjd_batch* b, int range)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_selfsync_range", "null batch");
    if (range < 0 || range > HJD_SS_FIX_MAXR || (range & 31))
        return fail(HJD_ERR_ARG, "hjd_batch_set_selfsync_range", "range must be 0 or a multiple of 32 up to HJD_SS_FIX_MAXR");
    b->ss_range_req = (uint32_t)range;
    return HJD_OK;
}

// Kernel 1b for the restart-free images of one chunk (see selfsync.cu).  Everything is enqueued on `st`; the
// synchronisation rounds terminate on the device, so the host never waits here.
static int run_selfsync(hjd_batch* b, const Chunk& c, size_t chunk_index, cudaStream_t st)
{
    if (c.ss1 <= c.ss0) return HJD_OK;
    const uint8_t* arena = (const uint8_t*)b->d_arena.p;
    const HjdImageDesc* imgs = (const HjdImageDesc*)b->d_imgs.p;
    const HjdTableSet* tsets = (const HjdTableSet*)b->d_tsets.p;
    const HjdSsImage* ss = (const HjdSsImage*)b->d_ss.p;
    const HjdSsWork* work = (const HjdSsWork*)b->d_sswork.p + c.sw0;
    const HjdSsWork* work_fix = (const HjdSsWork*)b->d_sswork.p + c.sf0;
    const int n_work = (int)(c.sw1 - c.sw0), n_work_fix = (int)(c.sf1 - c.sf0);
    const HjdSsSeg* segs = (const HjdSsSeg*)b->d_sssegs.p;
    uint8_t* dst = (uint8_t*)b->d_destuff.p;
    uint32_t* dlen = (uint32_t*)b->d_dlen.p;
    uint64_t* E = (uint64_t*)b->d_ssE0.p;
    uint64_t* X = (uint64_t*)b->d_ssX.p;
    uint32_t* tmp = (uint32_t*)b->d_scantmp.p + chunk_index * b->plan.ss_tmp_stride;
    uint32_t* ctl = (uint32_t*)b->d_flag.p + 4 * chunk_index;    // barrier count, last round with work, rounds run, item counter
    // [4][n_subs] (+ sentinel) counters of this chunk: starts, DC sums Y / Cb / Cr.  The kernels index them with
    // batch-wide sub-sequence numbers, hence the pointer that is shifted back by the chunk's first one.
    const uint32_t N = c.n_subs;
    uint32_t* cnt_region = (uint32_t*)b->d_ssnb.p + 4 * (size_t)c.sub0;
    uint32_t* cnt = cnt_region - c.sub0;

    CU(cudaMemsetAsync(ctl, 0, 4 * sizeof(uint32_t), st));
    CU(cudaMemsetAsync(cnt_region + 4 * (size_t)N, 0, sizeof(uint32_t), st));
    CU(hjd_launch_destuff(arena, imgs, ss + c.ss0, (int)(c.ss1 - c.ss0), c.ck0, c.n_ck, (uint32_t*)b->d_counts.p, tmp,
                          dst, dlen + c.ss0, st));
    b->launches += 2 + (c.n_ck + 1 > 2048 ? 3 : 1);
    CU(hjd_launch_ss_spec(imgs, tsets, ss, work, segs, n_work, dst, dlen, N, E, X, cnt, st));
    // a chain of wrong entry states can cross one range per round at worst: ranges + a confirming round
    const uint32_t max_rounds = N / 32 + 8;
    CU(hjd_launch_ss_sync(imgs, tsets, ss, work_fix, segs, n_work_fix, dst, dlen, N, E, X, cnt, ctl, max_rounds,
                          b->max_sync_ctas, st));
    CU(hjd_scan_u32(cnt_region, 4 * N + 1, tmp, st));                             // the counters become their exclusive prefix
    CU(hjd_launch_ss_write(imgs, tsets, ss, work, segs, n_work, dst, dlen, N, X, cnt, (int16_t*)b->d_coef.p,
                           (int32_t*)b->d_status.p, st));
    CU(hjd_launch_ss_fill_tail(imgs, ss + c.ss0, (int)(c.ss1 - c.ss0), cnt, (int16_t*)b->d_coef.p, st));
    b->launches += 4 + (4 * N + 1 > 2048 ? 3 : 1);
    b->ss_ran = true;
    return HJD_OK;
}

// Which fused kernel decodes a chunk's MCUs.  The tensor-core kernel (csrc/mcu_tc.cuh) is the faster one where its 128-MCU
// units are full and an MCU has several blocks to pipeline: large colour images (config 2: 3.39 ms against 3.63 ms, and the
// same time at every quality where the CUDA-core kernel's depends on the coefficients: 3.42 against 3.83 ms at q95; config 4:
// 0.221 against 0.242 ms).  Batches of small images are faster on the CUDA-core kernel (8192 thumbnails: 0.92 ms against
// 2.3 ms: a unit's set-up and pipeline fill are not amortised over one or two steps).
static int mcu_variant(unsigned flags, uint64_t blocks, uint32_t n_mcus, uint32_t n_images)
{
    if (flags & HJD_FLAG_TENSOR_CORE_IDCT) return HJD_MCU_TENSOR_CORE;
    if (flags & HJD_FLAG_CUDA_CORE_IDCT) return HJD_MCU_CUDA_CORE;
    // at least three blocks per MCU, at least eight full units per image, at least one unit for every group of every SM's CTA
    return (blocks >= 3ull * n_mcus && (uint64_t)n_mcus >= 1024ull * n_images && n_mcus >= 148u * 4u * 128u) ? HJD_MCU_TENSOR_CORE : HJD_MCU_CUDA_CORE;
}

// HJD_FLAG_EXIF_ORIENT: the orientation pass over the chunk's oriented images, from their staging regions to their
// places in the slab, right after the kernel that wrote them (counted in that kernel's stage).
static int launch_orient(hjd_batch* b, const Chunk& c, cudaStream_t st)
{
    if (c.oj1 <= c.oj0) return HJD_OK;
    const std::vector<uint32_t>& tiles = b->plan.orient_tiles;
    CU(hjd_launch_orient((uint8_t*)b->d_rgb.p, (const HjdOrientJob*)b->d_ojobs.p + c.oj0, (const uint32_t*)b->d_otiles.p + c.oj0,
                         (int)(c.oj1 - c.oj0), tiles[c.oj1] - tiles[c.oj0], (b->flags & HJD_FLAG_GRAY_OUT) ? 1 : 3, st));
    b->launches += 1;
    return HJD_OK;
}

// Kernels of one chunk on one stream.  ev != nullptr: record stage boundaries (serial mode only).
static int launch_chunk(hjd_batch* b, const Chunk& c, size_t chunk_index, cudaStream_t st, cudaEvent_t* ev)
{
    const uint8_t* arena = (const uint8_t*)b->d_arena.p;
    const HjdImageDesc* imgs = (const HjdImageDesc*)b->d_imgs.p;
    int32_t* status = (int32_t*)b->d_status.p;
    const int n = c.img1 - c.img0;
    if (!(b->flags & HJD_FLAG_HOST_SCAN) && n > 0) {
        CU(hjd_launch_marker_scan(arena, imgs, (uint32_t*)b->d_istart.p, status, c.img0, n,
                                  (const HjdScanSlice*)b->d_slices.p + c.slice0, (int)(c.slice1 - c.slice0),
                                  (uint32_t*)b->d_slicecnt.p + c.slice0, st));
        b->launches += 1 + (c.slice1 > c.slice0 ? 2 : 0);
    }
    if (ev) CU(cudaEventRecord(ev[1], st));
    {
        int rc = run_selfsync(b, c, chunk_index, st);      // counted in the entropy stage
        if (rc) return rc;
    }
    if (c.work1 > c.work0) {
        CU(hjd_launch_entropy_restart(arena, imgs, (const HjdTableSet*)b->d_tsets.p, (const uint32_t*)b->d_istart.p,
                                      (const HjdEntropyWork*)b->d_work.p + c.work0, (const HjdEntropySeg*)b->d_segs.p,
                                      (int)(c.work1 - c.work0),
                                      b->plan.max_tabs, (int16_t*)b->d_coef.p, status, st));
        b->launches += 1;
    }
    // multi-scan images: nothing else writes their blocks, and refinement scans read what the levels below left
    for (const auto& z : c.ms_zero)
        CU(cudaMemsetAsync((int16_t*)b->d_coef.p + z.first * 64, 0, z.second * 128, st));
    for (const auto& lv : c.ms_levels) {
        CU(hjd_launch_multiscan(arena, imgs, (const HjdScanDesc*)b->d_scans.p, (const HjdMsWork*)b->d_mswork.p + lv.first,
                                (int)(lv.second - lv.first), (const uint32_t*)b->d_msstarts.p,
                                (const HjdHuffTable*)b->d_mstabs.p, (int16_t*)b->d_coef.p, status, st));
        b->launches += 1;
    }
    if (ev) CU(cudaEventRecord(ev[2], st));
    if (!(b->flags & HJD_FLAG_KEEP_PLANES)) {
        // one output kernel in place of kernels 2+3, planes never reach HBM: luma-only (HJD_FLAG_GRAY_OUT) and reduced-size
        // (HJD_FLAG_SCALE_*) decodes have their own, the default is the fused kernel on the CUDA or the tensor cores
        if (c.blocks) {
            const int16_t* coef = (const int16_t*)b->d_coef.p;
            const HjdQuantSet* qsets = (const HjdQuantSet*)b->d_qsets.p;
            uint8_t* out = (uint8_t*)b->d_rgb.p;
            const uint32_t* mcu_prefix = (const uint32_t*)b->d_mcucta.p + c.img0;
            const uint32_t n_mcus = b->plan.mcu_cta[c.img1] - b->plan.mcu_cta[c.img0];
            const bool gray = (b->flags & HJD_FLAG_GRAY_OUT) != 0;
            const int shift = scale_shift(b->flags);
            if (gray) b->gy_chunks++;
            if (shift) {
                b->sc_chunks++;
                CU(hjd_launch_scaled(coef, imgs + c.img0, qsets, out, mcu_prefix, n, n_mcus, c.max_mcus, shift, gray, st));
            } else if (gray) {
                CU(hjd_launch_luma(coef, imgs + c.img0, qsets, out, (const uint32_t*)b->d_lumacta.p + c.img0, n,
                                   b->plan.luma_cta[c.img1] - b->plan.luma_cta[c.img0], c.max_luma, st));
            } else {
                const int variant = mcu_variant(b->flags, c.blocks, n_mcus, (uint32_t)n);
                if (variant == HJD_MCU_TENSOR_CORE) b->tc_chunks++; else b->cc_chunks++;
                CU(hjd_launch_mcu_rgb(coef, imgs + c.img0, qsets, out, mcu_prefix, n, n_mcus, c.max_mcus,
                                      (b->flags & HJD_FLAG_BMP_OUT) != 0, variant, st));
            }
            b->launches += 1;       // one even where the (image, CTA) grid takes several launches of 65,535 images
        }
        if (int rc = launch_orient(b, c, st)) return rc;
        if (ev) CU(cudaEventRecord(ev[3], st));
    } else {
        if (c.blocks) {
            CU(hjd_launch_idct_planes((const int16_t*)b->d_coef.p, imgs + c.img0, (const HjdQuantSet*)b->d_qsets.p,
                                      (uint8_t*)b->d_planes.p, n, c.max_blocks, st));
            b->launches += (n + 65534) / 65535;
        }
        if (ev) CU(cudaEventRecord(ev[3], st));
        if (c.blocks) {
            CU(hjd_launch_color((const uint8_t*)b->d_planes.p, imgs + c.img0, (uint8_t*)b->d_rgb.p, n, c.max_w, c.max_h, st));
            b->launches += (n + 65534) / 65535;
        }
        if (int rc = launch_orient(b, c, st)) return rc;       // the colour kernel writes the output here
    }
    return HJD_OK;
}

// All chunks: optional H2D of the files, kernels, optional D2H of the RGB region into rgb_host.
static int run_chunks(hjd_batch* b, bool h2d, uint8_t* rgb_host)
{
    cudaStream_t main = b->stream;
    b->launches = 0;
    b->tc_chunks = b->cc_chunks = b->sc_chunks = b->gy_chunks = 0;
    b->ss_ran = false;
    if (b->plan.any_parse_error && b->plan.rgb_bytes) CU(cudaMemsetAsync(b->d_rgb.p, 0, b->plan.rgb_bytes, main));
    CU(cudaEventRecord(b->ev[0], main));
    if (b->plan.chunks.size() <= 1) {
        // serial: one stream, stage boundaries recorded
        if (b->plan.chunks.empty()) {
            for (int k = 1; k <= 3; k++) CU(cudaEventRecord(b->ev[k], main));
        } else {
            const Chunk& c = b->plan.chunks[0];
            if (h2d) { int rc = copy_files(b, c, main); if (rc) return rc; CU(cudaEventRecord(b->ev[0], main)); }
            int rc = launch_chunk(b, c, 0, main, b->ev);
            if (rc) return rc;
        }
        CU(cudaEventRecord(b->ev[4], main));
        if (rgb_host && b->plan.rgb_bytes) CU(cudaMemcpyAsync(rgb_host, b->d_rgb.p, b->plan.rgb_bytes, cudaMemcpyDeviceToHost, main));
        return HJD_OK;
    }
    for (int k = 1; k <= 3; k++) CU(cudaEventRecord(b->ev[k], main));     // no per-stage times when chunks overlap
    CU(cudaEventRecord(b->ev_fork, main));
    for (int s = 0; s < HJD_NSTREAMS; s++) CU(cudaStreamWaitEvent(b->aux[s], b->ev_fork, 0));
    // From here on work is in flight on the chunk streams: whatever fails below, they are joined back into
    // the main stream before returning, so that the next upload (which synchronises only the main
    // stream before it rewrites the slabs) cannot overtake them.
    int rc_all = HJD_OK;
    for (size_t k = 0; k < b->plan.chunks.size() && rc_all == HJD_OK; k++) {
        const Chunk& c = b->plan.chunks[k];
        cudaStream_t st = b->aux[k % HJD_NSTREAMS];
        if (h2d) rc_all = copy_files(b, c, st);
        if (rc_all == HJD_OK) rc_all = launch_chunk(b, c, k, st, nullptr);
        if (rc_all == HJD_OK && rgb_host && c.rgb_hi > c.rgb_lo) {
            cudaError_t e = cudaMemcpyAsync(rgb_host + c.rgb_lo, (const uint8_t*)b->d_rgb.p + c.rgb_lo, c.rgb_hi - c.rgb_lo,
                                            cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) rc_all = fail(HJD_ERR_CUDA, "cudaMemcpyAsync (RGB chunk)", cudaGetErrorString(e));
        }
    }
    for (int s = 0; s < HJD_NSTREAMS; s++) {
        cudaError_t e = cudaEventRecord(b->ev_join[s], b->aux[s]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(main, b->ev_join[s], 0);
        if (e != cudaSuccess) {
            cudaStreamSynchronize(b->aux[s]);                    // last resort: wait here
            if (rc_all == HJD_OK) rc_all = fail(HJD_ERR_CUDA, "joining the chunk streams", cudaGetErrorString(e));
        }
    }
    if (rc_all != HJD_OK) return rc_all;
    CU(cudaEventRecord(b->ev[4], main));
    return HJD_OK;
}

extern "C" int hjd_batch_decode(hjd_batch* b)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_decode", "null batch");
    if (!b->uploaded) return fail(HJD_ERR_STATE, "hjd_batch_decode", "nothing uploaded");
    CU(cudaSetDevice(b->device));
    int rc = run_chunks(b, false, nullptr);
    if (rc) return rc;
    b->decoded = true;
    return HJD_OK;
}

extern "C" int hjd_batch_sync(hjd_batch* b)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_sync", "null batch");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

extern "C" int hjd_batch_num_images(const hjd_batch* b) { return b ? (int)b->plan.imgs.size() : 0; }
extern "C" int hjd_batch_idct_variant(const hjd_batch* b)
{
    if (!b || (b->flags & HJD_FLAG_KEEP_PLANES)) return 0;
    return (b->tc_chunks ? 1 : 0) | (b->cc_chunks ? 2 : 0) | (b->sc_chunks ? 4 : 0) | (b->gy_chunks ? 8 : 0);
}
// Kernel 1b's round words of the last decode (run_selfsync), read once the stream is idle: the most rounds any chunk
// ran (working rounds + the one that confirmed), and whether a chunk hit the round limit.
static cudaError_t selfsync_control(const hjd_batch* b, uint32_t* most, bool* hit_limit)
{
    const std::vector<Chunk>& chunks = b->plan.chunks;
    std::vector<uint32_t> ctl(4 * chunks.size() + 4, 0);
    const cudaError_t e = cudaMemcpy(ctl.data(), b->d_flag.p, 4 * chunks.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    *most = 0;
    *hit_limit = false;
    for (size_t k = 0; k < chunks.size(); k++) {
        if (chunks[k].ss1 <= chunks[k].ss0) continue;
        if ((ctl[4 * k + 2] & 0x7FFFFFFFu) > *most) *most = ctl[4 * k + 2] & 0x7FFFFFFFu;
        if (ctl[4 * k + 2] & 0x80000000u) *hit_limit = true;
    }
    return e;
}

extern "C" int hjd_batch_selfsync_rounds(hjd_batch* b)
{
    // rounds the device-side loop ran in the last decode, in the chunk that needed the most; syncs
    if (!b || !b->ss_ran || !b->d_flag.p) return 0;
    uint32_t most;
    bool hit_limit;
    if (cudaSetDevice(b->device) != cudaSuccess || cudaStreamSynchronize(b->stream) != cudaSuccess ||
        selfsync_control(b, &most, &hit_limit) != cudaSuccess) { cudaGetLastError(); return -1; }
    return (int)most;
}

extern "C" int hjd_batch_get_info(const hjd_batch* b, int i, hjd_image_info* o)
{
    if (!b || !o || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_get_info", "bad arguments");
    const HjdImageDesc& d = b->plan.imgs[i];
    memset(o, 0, sizeof *o);
    o->width = d.width; o->height = d.height; o->ncomp = d.ncomp; o->hf = d.hf; o->vf = d.vf;
    o->blocks_per_mcu = d.blocks_per_mcu; o->mcus_x = d.mcus_x; o->mcus_y = d.mcus_y;
    o->restart_interval = d.restart_interval; o->n_intervals = d.n_intervals; o->scan_bytes = d.scan_len;
    o->block_base = d.block_base; o->n_blocks = d.n_blocks; o->rgb_offset = b->plan.out_off[i];
    o->y_offset = d.y_off; o->cb_offset = d.cb_off; o->cr_offset = d.cr_off;
    o->y_pitch = d.y_pitch; o->c_pitch = d.c_pitch; o->status = b->plan.parse_status[i];
    if (b->plan.ms_items[i]) o->n_intervals = b->plan.ms_items[i];
    return HJD_OK;
}

extern "C" int hjd_batch_get_out_size(const hjd_batch* b, int i, uint32_t* w, uint32_t* h)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_get_out_size", "bad arguments");
    const HjdImageDesc& d = b->plan.imgs[i];
    uint32_t ow, oh;
    out_size(b->flags, d.width, d.height, b->plan.orientation[i], &ow, &oh);
    if (w) *w = ow;
    if (h) *h = oh;
    return HJD_OK;
}

extern "C" int hjd_batch_get_orientation(const hjd_batch* b, int i)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_get_orientation", "bad arguments");
    return b->plan.orientation[i];
}

extern "C" int hjd_batch_num_scans(const hjd_batch* b, int i)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_num_scans", "bad arguments");
    return (int)b->plan.n_scans[i];
}

extern "C" int hjd_batch_get_status(hjd_batch* b, int32_t* status)
{
    if (!b || !status) return fail(HJD_ERR_ARG, "hjd_batch_get_status", "bad arguments");
    CU(cudaSetDevice(b->device));
    const size_t n = b->plan.imgs.size();
    if (n == 0) return HJD_OK;
    CU(cudaMemcpyAsync(status, b->d_status.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    if (b->ss_ran) {       // the device-side synchronisation loop reports here if it ever hit its round limit
        uint32_t most;
        bool hit_limit;
        CU(selfsync_control(b, &most, &hit_limit));
        if (hit_limit) return fail(HJD_ERR_STATE, "self-synchronising decode", "did not converge");
    }
    for (size_t i = 0; i < n; i++) {
        if (b->plan.parse_status[i] != 0) status[i] = b->plan.parse_status[i];
        else if (b->plan.host_restart_warn[i]) status[i] |= HJD_IMG_WARN_RESTART;
    }
    return HJD_OK;
}

extern "C" int hjd_batch_get_timings(hjd_batch* b, hjd_timings* t)
{
    if (!b || !t) return fail(HJD_ERR_ARG, "hjd_batch_get_timings", "bad arguments");
    if (!b->decoded) return fail(HJD_ERR_STATE, "hjd_batch_get_timings", "no decode yet");
    CU(cudaSetDevice(b->device));
    CU(cudaEventSynchronize(b->ev[4]));
    CU(cudaEventElapsedTime(&t->scan_ms, b->ev[0], b->ev[1]));
    CU(cudaEventElapsedTime(&t->entropy_ms, b->ev[1], b->ev[2]));
    CU(cudaEventElapsedTime(&t->idct_ms, b->ev[2], b->ev[3]));
    CU(cudaEventElapsedTime(&t->color_ms, b->ev[3], b->ev[4]));
    CU(cudaEventElapsedTime(&t->total_ms, b->ev[0], b->ev[4]));
    t->launches = b->launches;
    return HJD_OK;
}

extern "C" int hjd_batch_mark(hjd_batch* b, int slot)
{
    if (!b || slot < 0 || slot >= HJD_MARK_SLOTS) return fail(HJD_ERR_ARG, "hjd_batch_mark", "bad arguments");
    CU(cudaSetDevice(b->device));
    CU(cudaEventRecord(b->mark[slot], b->stream));
    return HJD_OK;
}

extern "C" float hjd_batch_elapsed_ms(hjd_batch* b, int slot_a, int slot_b)
{
    if (!b || slot_a < 0 || slot_a >= HJD_MARK_SLOTS || slot_b < 0 || slot_b >= HJD_MARK_SLOTS) { fail(HJD_ERR_ARG, "hjd_batch_elapsed_ms", "bad arguments"); return -1.f; }
    float ms = -1.f;
    if (cudaSetDevice(b->device) != cudaSuccess || cudaEventSynchronize(b->mark[slot_b]) != cudaSuccess ||
        cudaEventElapsedTime(&ms, b->mark[slot_a], b->mark[slot_b]) != cudaSuccess) {
        fail(HJD_ERR_CUDA, "hjd_batch_elapsed_ms", cudaGetErrorString(cudaGetLastError()));
        return -1.f;
    }
    return ms;
}

extern "C" uint64_t hjd_batch_rgb_bytes(const hjd_batch* b)   { return b ? b->plan.rgb_bytes : 0; }
extern "C" uint64_t hjd_batch_coef_bytes(const hjd_batch* b)  { return b ? b->plan.total_blocks * 128 : 0; }
extern "C" uint64_t hjd_batch_plane_bytes(const hjd_batch* b) { return b ? b->plan.plane_bytes : 0; }
extern "C" uint64_t hjd_batch_scan_bytes(const hjd_batch* b)  { return b ? b->plan.scan_bytes : 0; }
extern "C" uint64_t hjd_batch_pixels(const hjd_batch* b)      { return b ? b->plan.pixels : 0; }
extern "C" void* hjd_batch_device_rgb(hjd_batch* b)    { return b ? b->d_rgb.p : nullptr; }
extern "C" void* hjd_batch_device_coef(hjd_batch* b)   { return b ? b->d_coef.p : nullptr; }
extern "C" void* hjd_batch_device_planes(hjd_batch* b) { return b ? b->d_planes.p : nullptr; }

static int download(hjd_batch* b, void* dst, const void* src, uint64_t bytes, const char* who)
{
    if (!b || !dst) return fail(HJD_ERR_ARG, who, "bad arguments");
    if (!b->decoded) return fail(HJD_ERR_STATE, who, "no decode yet");
    CU(cudaSetDevice(b->device));
    if (bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

extern "C" int hjd_batch_download_rgb(hjd_batch* b, uint8_t* dst)
{ return download(b, dst, b ? b->d_rgb.p : nullptr, b ? b->plan.rgb_bytes : 0, "hjd_batch_download_rgb"); }

extern "C" int hjd_batch_download_image(hjd_batch* b, int i, uint8_t* dst)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_image", "bad arguments");
    if (b->flags & HJD_FLAG_BMP_OUT) return fail(HJD_ERR_STATE, "hjd_batch_download_image", "this batch writes BMP files (HJD_FLAG_BMP_OUT): use hjd_batch_download_bmp");
    const HjdImageDesc& d = b->plan.imgs[i];
    return download(b, dst, (const uint8_t*)b->d_rgb.p + b->plan.out_off[i], image_out_bytes(b->flags, d.width, d.height),
                    "hjd_batch_download_image");
}

extern "C" uint64_t hjd_batch_bmp_bytes(const hjd_batch* b, int i)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size() || !(b->flags & HJD_FLAG_BMP_OUT) || b->plan.parse_status[i] != HJD_IMG_OK) return 0;
    const HjdImageDesc& d = b->plan.imgs[i];
    return 54 + (uint64_t)((d.width * 3 + 3) & ~3u) * d.height;                  // openjpg.cpp:541
}

extern "C" int hjd_batch_download_bmp(hjd_batch* b, int i, uint8_t* dst)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_bmp", "bad arguments");
    if (!(b->flags & HJD_FLAG_BMP_OUT)) return fail(HJD_ERR_STATE, "hjd_batch_download_bmp", "batch was not created with HJD_FLAG_BMP_OUT");
    return download(b, dst, (const uint8_t*)b->d_rgb.p + b->plan.out_off[i] + 10, hjd_batch_bmp_bytes(b, i), "hjd_batch_download_bmp");
}

extern "C" int hjd_batch_download_coef(hjd_batch* b, int16_t* dst)
{ return download(b, dst, b ? b->d_coef.p : nullptr, b ? b->plan.total_blocks * 128 : 0, "hjd_batch_download_coef"); }

extern "C" int hjd_batch_download_image_coef(hjd_batch* b, int i, int16_t* dst)
{
    if (!b || i < 0 || i >= (int)b->plan.imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_image_coef", "bad arguments");
    const HjdImageDesc& d = b->plan.imgs[i];
    return download(b, dst, (const uint8_t*)b->d_coef.p + d.block_base * 128, d.n_blocks * 128, "hjd_batch_download_image_coef");
}

extern "C" int hjd_batch_download_planes(hjd_batch* b, uint8_t* dst)
{
    if (b && !(b->flags & HJD_FLAG_KEEP_PLANES)) return fail(HJD_ERR_STATE, "hjd_batch_download_planes", "planes exist in HBM only with HJD_FLAG_KEEP_PLANES (the default kernels keep them in shared memory)");
    return download(b, dst, b ? b->d_planes.p : nullptr, b ? b->plan.plane_bytes : 0, "hjd_batch_download_planes");
}

// ------------------------------------------------------------------------------------------
// host-buffer end-to-end path
// ------------------------------------------------------------------------------------------
extern "C" uint64_t hjd_out_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n, unsigned flags)
{
    uint64_t total = 0;
    if (!arena || !offsets || !sizes) return 0;
    HjdParsed ps;
    std::unique_ptr<HjdMultiParsed> mp;
    for (int i = 0; i < n; i++) {
        int st = hjd_parse_jpeg(arena + offsets[i], (size_t)sizes[i], &ps);
        if (st == HJD_IMG_ERR_UNSUPPORTED && (flags & HJD_FLAG_MULTI_SCAN)) {
            if (!mp) mp.reset(new HjdMultiParsed());
            st = hjd_parse_jpeg_multi(arena + offsets[i], (size_t)sizes[i], mp.get());
            ps = mp->frame;
        }
        if (st == HJD_IMG_OK) total += align_up(image_out_bytes(flags, ps.width, ps.height), 256);
    }
    return total;
}

extern "C" uint64_t hjd_rgb_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n)
{ return hjd_out_slab_bytes(arena, offsets, sizes, n, 0); }

extern "C" int hjd_batch_decode_host(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes,
                                     int n, uint8_t* rgb_out, uint64_t rgb_capacity, uint64_t* rgb_offsets_out,
                                     int32_t* status_out, int chunk_images)
{
    if (!b || !arena || !offsets || !sizes || !rgb_out || n < 0 || chunk_images < 0) return fail(HJD_ERR_ARG, "hjd_batch_decode_host", "bad arguments");
    CU(cudaSetDevice(b->device));
    b->chunk_images = chunk_images;                               // 0: chunks planned from the block counts (see plan_chunks)
    int rc = prepare_arena(b, arena, offsets, sizes, n, true);    // parse + metadata; files not copied yet
    b->chunk_images = 0;
    if (rc) return rc;
    if (b->plan.rgb_bytes > rgb_capacity) return fail(HJD_ERR_ARG, "hjd_batch_decode_host", "rgb_out too small");
    rc = run_chunks(b, true, rgb_out);                            // per chunk: H2D, kernels, D2H
    if (rc) return rc;
    b->decoded = true;
    if (rgb_offsets_out)
        for (int i = 0; i < n; i++) rgb_offsets_out[i] = b->plan.out_off[i];
    if (status_out) { rc = hjd_batch_get_status(b, status_out); if (rc) return rc; }
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

// NUMA node of a GPU (from sysfs via its PCI address), -1 when the platform does not say.
static int device_numa_node(int device)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* p = bus; *p; p++) if (*p >= 'A' && *p <= 'F') *p = (char)(*p - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* fp = fopen(path, "r");
    if (!fp) return -1;
    int node = -1;
    if (fscanf(fp, "%d", &node) != 1) node = -1;
    fclose(fp);
    return node;
}

extern "C" int hjd_device_numa_node(int device) { return device_numa_node(device); }

// Pinned host memory whose pages come from the NUMA node next to `device` (set_mempolicy(MPOL_PREFERRED)
// around the allocation: cudaHostAlloc faults the pages in on the calling thread).  The D2H copy of a
// decoded batch is the end-to-end bottleneck, and a buffer on the far socket halves it on two-socket
// hosts.  Falls back to plain hjd_host_alloc when the platform exposes no NUMA topology.
extern "C" void* hjd_host_alloc_near(int device, size_t bytes)
{
    const int node = device_numa_node(device);
    bool bound = false;
#ifdef SYS_set_mempolicy
    if (node >= 0 && node < 1024) {
        unsigned long mask[16];
        memset(mask, 0, sizeof mask);
        mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
        bound = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(sizeof mask * 8)) == 0;
    }
#endif
    void* p = hjd_host_alloc(bytes);
#ifdef SYS_set_mempolicy
    if (bound) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
#endif
    (void)bound;
    return p;
}

// Raw link probe: `reps` times, concurrently on two streams and with no kernel anywhere, h2d_bytes from
// host_in to the device and d2h_bytes from the device to host_out (both pinned).  *ms = wall time of the
// slower direction per repetition.  This is the ceiling hjd_batch_decode_host works against.
extern "C" int hjd_link_probe(int device, const void* host_in, size_t h2d_bytes, void* host_out, size_t d2h_bytes,
                              int reps, float* ms_h2d, float* ms_d2h)
{
    if (reps <= 0) return fail(HJD_ERR_ARG, "hjd_link_probe", "bad arguments");
    CU(cudaSetDevice(device));
    void *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int rc = HJD_OK;
    auto cleanup = [&]() {
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        for (auto& q : s) if (q) cudaStreamDestroy(q);
        if (d_in) cudaFree(d_in);
        if (d_out) cudaFree(d_out);
    };
    cudaError_t e = cudaSuccess;
    if (h2d_bytes && host_in) e = cudaMalloc(&d_in, h2d_bytes);
    if (e == cudaSuccess && d2h_bytes && host_out) e = cudaMalloc(&d_out, d2h_bytes);
    for (int k = 0; k < 2 && e == cudaSuccess; k++) e = cudaStreamCreateWithFlags(&s[k], cudaStreamNonBlocking);
    for (int k = 0; k < 4 && e == cudaSuccess; k++) e = cudaEventCreate(&ev[k]);
    if (e == cudaSuccess && d_out) e = cudaMemset(d_out, 0x5a, d2h_bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        cudaEventRecord(ev[0], s[0]); cudaEventRecord(ev[2], s[1]);
        for (int r = 0; r < reps; r++) {
            if (d_in) cudaMemcpyAsync(d_in, host_in, h2d_bytes, cudaMemcpyHostToDevice, s[0]);
            if (d_out) cudaMemcpyAsync(host_out, d_out, d2h_bytes, cudaMemcpyDeviceToHost, s[1]);
        }
        cudaEventRecord(ev[1], s[0]); cudaEventRecord(ev[3], s[1]);
        e = cudaStreamSynchronize(s[0]);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s[1]);
        float a = 0.f, b = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&a, ev[0], ev[1]);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&b, ev[2], ev[3]);
        if (ms_h2d) *ms_h2d = a / (float)reps;
        if (ms_d2h) *ms_d2h = b / (float)reps;
    }
    if (e != cudaSuccess) rc = fail(HJD_ERR_CUDA, "hjd_link_probe", cudaGetErrorString(e));
    cleanup();
    return rc;
}

extern "C" void* hjd_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); fail(HJD_ERR_NOMEM, "cudaHostAlloc"); return nullptr; }
    return p;
}
extern "C" void hjd_host_free(void* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------
// reference-shaped single-image calls
// ------------------------------------------------------------------------------------------
struct DefaultBatch {
    hjd_batch* b[2] = {nullptr, nullptr};      // [0] RGB out (DecodeJpgFileData), [1] BMP out (ConvertJpgFile)
    int device[2] = {-1, -1};
    ~DefaultBatch() { for (int k = 0; k < 2; k++) if (b[k]) hjd_batch_destroy(b[k]); }
};
static thread_local DefaultBatch g_default;
static std::atomic<int> g_default_device(0);

extern "C" int hjd_set_default_device(int device)
{
    if (device < 0 || device >= hjd_device_count()) return fail(HJD_ERR_ARG, "hjd_set_default_device", "bad device index");
    g_default_device.store(device);
    return HJD_OK;
}

// The lazily created per-thread batch behind the single-image calls, on the process-wide default device.
static hjd_batch* default_batch(bool bmp)
{
    const int k = bmp ? 1 : 0, dev = g_default_device.load();
    if (g_default.b[k] && g_default.device[k] != dev) { hjd_batch_destroy(g_default.b[k]); g_default.b[k] = nullptr; }
    if (!g_default.b[k]) { g_default.b[k] = hjd_batch_create(dev, bmp ? HJD_FLAG_BMP_OUT : 0); g_default.device[k] = dev; }
    return g_default.b[k];
}

extern "C" void hjd_free(void* p) { free(p); }

extern "C" int hjd_get_image_size(const uint8_t* buf, int size, unsigned* width, unsigned* height)
{
    HjdParsed ps;
    if (!buf || size <= 0 || hjd_parse_jpeg(buf, (size_t)size, &ps) != HJD_IMG_OK) { fail(HJD_ERR_ARG, "hjd_get_image_size", "not a decodable baseline JPEG"); return 0; }
    if (width) *width = ps.width;
    if (height) *height = ps.height;
    return 1;
}

static void fill_info_from_parse(const HjdParsed& ps, hjd_image_info* o)
{
    memset(o, 0, sizeof *o);
    o->status = ps.status;
    if (ps.status != HJD_IMG_OK) return;
    const FrameGeometry g = frame_geometry(ps.width, ps.height, ps.ncomp, ps.hf, ps.vf, ps.restart_interval);
    o->width = ps.width; o->height = ps.height; o->ncomp = (uint8_t)ps.ncomp; o->hf = (uint8_t)ps.hf; o->vf = (uint8_t)ps.vf;
    o->blocks_per_mcu = (uint8_t)g.blocks_per_mcu; o->mcus_x = g.mcus_x; o->mcus_y = g.mcus_y;
    o->restart_interval = ps.restart_interval;
    o->n_intervals = g.n_intervals;
    o->scan_bytes = (uint32_t)ps.scan_len;
    o->n_blocks = (uint64_t)g.n_mcus * o->blocks_per_mcu;
}

extern "C" int hjd_probe_jpeg(const uint8_t* buf, int64_t size, hjd_image_info* out)
{
    HjdParsed ps;
    const int st = (buf && size > 0) ? hjd_parse_jpeg(buf, (size_t)size, &ps) : HJD_IMG_ERR_NOT_JPEG;
    if (buf && size > 0 && st == HJD_IMG_OK) {
        HjdTableSet ts;
        ps.status = hjd_build_table_set(ps, &ts);                  // an over-subscribed DHT is a per-image error too
    } else ps.status = st;
    if (out) fill_info_from_parse(ps, out);
    return ps.status;
}

// Multi-scan parse plus every table build: the status a batch with HJD_FLAG_MULTI_SCAN reports for the file.
static int probe_multi(const uint8_t* buf, int64_t size, HjdMultiParsed* mp)
{
    int st = hjd_parse_jpeg_multi(buf, (size_t)size, mp);
    if (st == HJD_IMG_OK && mp->frame.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
    HjdHuffTable t;
    for (size_t k = 0; st == HJD_IMG_OK && k < mp->scans.size(); k++) {
        const HjdScanParsed& s = mp->scans[k];
        for (int c = 0; c < s.ncomp; c++) {
            if (s.dc[c].present && !hjd_build_huff_table(s.dc[c], false, &t)) st = HJD_IMG_ERR_BAD_TABLE;
            if (s.ac[c].present && !(s.kind == HJD_SCAN_SEQ ? hjd_build_huff_table(s.ac[c], true, &t) : hjd_build_huff_table_raw(s.ac[c], &t)))
                st = HJD_IMG_ERR_BAD_TABLE;
        }
    }
    return mp->frame.status = st;
}

extern "C" int hjd_probe_jpeg_flags(const uint8_t* buf, int64_t size, unsigned flags, hjd_image_info* out)
{
    const int st = hjd_probe_jpeg(buf, size, out);
    if (st != HJD_IMG_ERR_UNSUPPORTED || !(flags & HJD_FLAG_MULTI_SCAN)) return st;
    std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
    probe_multi(buf, size, mp.get());
    const HjdParsed& f = mp->frame;
    if (out) {
        fill_info_from_parse(f, out);
        if (f.status == HJD_IMG_OK) {
            out->n_intervals = 0;
            for (const HjdScanParsed& s : mp->scans)
                if (scan_is_read(flags, s)) out->n_intervals += ms_scan_items(f, s, nullptr, nullptr);
        }
    }
    return f.status;
}

extern "C" int hjd_probe_jpeg_orientation(const uint8_t* buf, int64_t size)
{
    if (!buf || size < 2 || buf[0] != 0xFF || buf[1] != 0xD8) return HJD_IMG_ERR_NOT_JPEG;
    HjdParsed ps;
    if (hjd_parse_jpeg(buf, (size_t)size, &ps) != HJD_IMG_ERR_UNSUPPORTED) return ps.orientation;
    // e.g. a progressive file: the multi-scan walk, which does not stop at its SOF2, reads the Exif APP1 wherever it is
    std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
    hjd_parse_jpeg_multi(buf, (size_t)size, mp.get());
    return mp->frame.orientation;
}

extern "C" int hjd_probe_jpeg_scans(const uint8_t* buf, int64_t size, hjd_scan_info* out, int max)
{
    if (max < 0 || (max > 0 && !out)) return fail(HJD_ERR_ARG, "hjd_probe_jpeg_scans", "bad arguments");
    hjd_image_info info;
    const int st = hjd_probe_jpeg(buf, size, &info);
    if (st == HJD_IMG_OK) {                       // one interleaved sequential scan
        if (max > 0) {
            memset(out, 0, sizeof *out);
            out->ncomp = info.ncomp;
            for (int c = 0; c < info.ncomp; c++) out->comp[c] = (uint8_t)c;
            out->se = 63;
            out->restart_interval = info.restart_interval;
            out->bytes = info.scan_bytes;
        }
        return 1;
    }
    if (st != HJD_IMG_ERR_UNSUPPORTED) return st;
    std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
    const int ms = probe_multi(buf, size, mp.get());
    if (ms != HJD_IMG_OK) return ms;
    for (int k = 0; k < (int)mp->scans.size() && k < max; k++) {
        const HjdScanParsed& s = mp->scans[(size_t)k];
        hjd_scan_info& o = out[k];
        memset(&o, 0, sizeof o);
        o.ncomp = (uint8_t)s.ncomp;
        for (int c = 0; c < s.ncomp; c++) o.comp[c] = (uint8_t)s.comp[c];
        o.ss = (uint8_t)s.ss; o.se = (uint8_t)s.se; o.ah = (uint8_t)s.ah; o.al = (uint8_t)s.al;
        o.level = (uint8_t)(s.level < 255 ? s.level : 255);
        o.restart_interval = s.restart_interval;
        o.bytes = (uint32_t)s.len;
    }
    return (int)mp->scans.size();
}

extern "C" uint32_t hjd_huff_lookup_probe(const uint8_t bits[16], const uint8_t* vals, int nvals, int is_ac, uint32_t peek16)
{
    static thread_local HjdHuffTable tab;
    static thread_local HjdRawHuff cached;
    static thread_local int cached_ac = -1;
    HjdRawHuff raw;
    memset(&raw, 0, sizeof raw);
    if (!bits || !vals || nvals < 0 || nvals > 256) return 0xFFFFFFFFu;
    memcpy(raw.bits, bits, 16);
    memcpy(raw.vals, vals, (size_t)nvals);
    raw.nvals = nvals;
    raw.present = 1;
    if (cached_ac != is_ac || memcmp(&cached, &raw, sizeof raw) != 0) {
        cached_ac = -1;
        if (!hjd_build_huff_table(raw, is_ac != 0, &tab)) return 0xFFFFFFFFu;
        cached = raw;
        cached_ac = is_ac;
    }
    return hjd_host_huff_lookup(&tab, peek16);
}

// One image through a default batch; the result (RGB24, or the BMP file) is downloaded into memory from
// alloc(bytes).  The staging is the batch's own pinned buffer: one asynchronous copy, one host copy.
static int decode_one(bool bmp, const uint8_t* buf, int size, void* (*alloc)(size_t), uint8_t** out_ptr, size_t* out_bytes,
                      unsigned* width, unsigned* height, const char* who)
{
    if (!buf || size <= 0 || !out_ptr || !alloc) { fail(HJD_ERR_ARG, who, "bad arguments"); return 0; }
    *out_ptr = nullptr;
    hjd_batch* b = default_batch(bmp);
    if (!b) return 0;
    const uint8_t* bufs[1] = {buf};
    const int64_t sizes[1] = {size};
    if (hjd_batch_upload(b, bufs, sizes, 1) != HJD_OK) return 0;
    if (b->plan.parse_status[0] != HJD_IMG_OK) { fail(HJD_ERR_ARG, who, "unsupported or corrupt JPEG"); return 0; }
    if (hjd_batch_decode(b) != HJD_OK) return 0;
    const HjdImageDesc& d = b->plan.imgs[0];
    const size_t bytes = bmp ? (size_t)hjd_batch_bmp_bytes(b, 0) : (size_t)d.width * d.height * 3;
    if (cudaSetDevice(b->device) != cudaSuccess || b->h_out.ensure(bytes + 16) != cudaSuccess) { cudaGetLastError(); fail(HJD_ERR_NOMEM, who, "pinned staging buffer"); return 0; }
    if (cudaMemcpyAsync(b->h_out.p, (const uint8_t*)b->d_rgb.p + b->plan.out_off[0] + (bmp ? 10 : 0), bytes, cudaMemcpyDeviceToHost, b->stream) != cudaSuccess ||
        cudaStreamSynchronize(b->stream) != cudaSuccess) { fail(HJD_ERR_CUDA, who, cudaGetErrorString(cudaGetLastError())); return 0; }
    uint8_t* out = (uint8_t*)alloc(bytes ? bytes : 1);
    if (!out) { fail(HJD_ERR_NOMEM, who, "allocation failed"); return 0; }
    memcpy(out, b->h_out.p, bytes);
    *out_ptr = out;
    if (out_bytes) *out_bytes = bytes;
    if (width) *width = d.width;
    if (height) *height = d.height;
    return 1;
}

extern "C" int hjd_decode_jpg_file_data_alloc(const uint8_t* buf, int size, void* (*alloc)(size_t), uint8_t** rgb,
                                              unsigned* width, unsigned* height)
{
    return decode_one(false, buf, size, alloc, rgb, nullptr, width, height, "hjd_decode_jpg_file_data");
}

extern "C" int hjd_decode_jpg_file_data(const uint8_t* buf, int size, uint8_t** rgb, unsigned* width, unsigned* height)
{
    return decode_one(false, buf, size, malloc, rgb, nullptr, width, height, "hjd_decode_jpg_file_data");
}

extern "C" size_t hjd_encode_bmp24(unsigned width, unsigned height, const uint8_t* rgb, uint8_t* out)
{
    // openjpg.cpp:504-570: 14+40 byte header, bottom-up, B G R, each row padded to a multiple of 4.
    const unsigned pad = (4 - (width * 3) % 4) % 4;
    const size_t total = (size_t)width * height * 3 + (size_t)height * pad + 54;
    if (!out) return total;
    memset(out, 0, 54);
    auto put32 = [&](int at, uint32_t v) { out[at] = v & 255; out[at + 1] = (v >> 8) & 255; out[at + 2] = (v >> 16) & 255; out[at + 3] = (v >> 24) & 255; };
    out[0] = 'B'; out[1] = 'M';
    put32(2, (uint32_t)total);
    put32(10, 54);
    put32(14, 40);
    put32(18, width);
    put32(22, height);
    out[26] = 1;
    out[28] = 24;
    uint8_t* o = out + 54;
    for (unsigned row = height; row-- > 0;) {
        const uint8_t* src = rgb + (size_t)row * width * 3;
        for (unsigned x = 0; x < width; x++) { o[0] = src[2]; o[1] = src[1]; o[2] = src[0]; o += 3; src += 3; }
        for (unsigned k = 0; k < pad; k++) *o++ = 0;
    }
    return total;
}

extern "C" int hjd_write_bmp24(const char* path, unsigned width, unsigned height, const uint8_t* rgb)
{
    if (!path || !rgb) { fail(HJD_ERR_ARG, "hjd_write_bmp24", "bad arguments"); return 0; }
    const size_t total = hjd_encode_bmp24(width, height, rgb, nullptr);
    uint8_t* tmp = (uint8_t*)malloc(total);
    if (!tmp) { fail(HJD_ERR_NOMEM, "malloc"); return 0; }
    hjd_encode_bmp24(width, height, rgb, tmp);
    FILE* fp = fopen(path, "wb");
    if (!fp) { free(tmp); fail(HJD_ERR_IO, "fopen", path); return 0; }
    const size_t w = fwrite(tmp, 1, total, fp);
    fclose(fp);
    free(tmp);
    if (w != total) { fail(HJD_ERR_IO, "fwrite", path); return 0; }
    return 1;
}

extern "C" int hjd_convert_jpg_file(const char* jpg_in, const char* bmp_out)
{
    // ConvertJpgFile, openjpg.cpp:593-684: returns 1 on success, 0 on failure.  The decode runs with
    // HJD_FLAG_BMP_OUT: what comes back from the GPU is the file WriteBMP24 would write.
    if (!jpg_in || !bmp_out) { fail(HJD_ERR_ARG, "hjd_convert_jpg_file", "bad arguments"); return 0; }
    FILE* fp = fopen(jpg_in, "rb");
    if (!fp) { fail(HJD_ERR_IO, "fopen", jpg_in); return 0; }          // openjpg.cpp:603-608
    fseek(fp, 0, SEEK_END);
    const long len = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    if (len <= 0 || len > 0x7FFFFFFF) { fclose(fp); fail(HJD_ERR_IO, "empty or oversized file", jpg_in); return 0; }
    uint8_t* buf = (uint8_t*)malloc((size_t)len);
    if (!buf) { fclose(fp); fail(HJD_ERR_NOMEM, "malloc"); return 0; }
    const size_t got = fread(buf, 1, (size_t)len, fp);
    fclose(fp);
    uint8_t* bmp = nullptr;
    size_t bytes = 0;
    int ok = (got == (size_t)len) && decode_one(true, buf, (int)len, malloc, &bmp, &bytes, nullptr, nullptr, "hjd_convert_jpg_file");
    free(buf);
    if (!ok) return 0;
    fp = fopen(bmp_out, "wb");
    if (!fp) { free(bmp); fail(HJD_ERR_IO, "fopen", bmp_out); return 0; }
    ok = fwrite(bmp, 1, bytes, fp) == bytes;
    if (fclose(fp) != 0) ok = 0;
    free(bmp);
    if (!ok) fail(HJD_ERR_IO, "fwrite", bmp_out);
    return ok;
}
