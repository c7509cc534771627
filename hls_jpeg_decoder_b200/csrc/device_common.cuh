// csrc/device_common.cuh -- small device helpers shared by the kernel files, and the grid policy of the per-image output
// kernels (hjd_k_mcu_rgb, hjd_k_luma, hjd_k_mcu_scaled).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

// Byte offset of the second-level table inside HjdHuffTable, for 32-bit shared-window addressing.
#define HJD_TAB_LUT2_OFF (HJD_LUT_SIZE * 2)

// Meaning of a decoded symbol (see HjdHuffTable); also used by the host when it fills the LUT.
__host__ __device__ __forceinline__ uint32_t hjd_sym_fields(uint32_t len, uint32_t sym, bool is_ac)
{
    const uint32_t size = sym & 15u, run = sym >> 4;
    if (!is_ac) return HJD_SYM_FIELDS(len, size, 1);                          // DC: loadjpg.cpp:616-667
    if (size) return HJD_SYM_FIELDS(len, size, run + 1);                      // loadjpg.cpp:778-806
    return HJD_SYM_FIELDS(len, 0, run == 0 ? 63 : (run == 15 ? 16 : 0));      // EOB / ZRL / ignored, 771-775
}

__device__ __forceinline__ uint32_t hjd_lds_u16(uint32_t a) { uint16_t v; asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t hjd_lds_u8(uint32_t a) { uint32_t v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t hjd_lds_u32(uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t hjd_lds_u16_sync(uint32_t a) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void hjd_sts_u16_sync(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "h"((uint16_t)v) : "memory"); }
__device__ __forceinline__ void hjd_sts_v2_sync(uint32_t a, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(a), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ uint2 hjd_lds_v2_sync(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint4 hjd_lds_v4_sync(uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void hjd_sts_zero16_sync(uint32_t a) { asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" :: "r"(a), "r"(0) : "memory"); }
// PTX shifts clamp the amount to 32 (result 0), unlike C++ where a shift by 32 is undefined.
__device__ __forceinline__ uint32_t hjd_shr(uint32_t v, uint32_t n) { uint32_t r; asm("shr.u32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n)); return r; }
__device__ __forceinline__ uint32_t hjd_shl(uint32_t v, uint32_t n) { uint32_t r; asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n)); return r; }


// The symbol whose code starts the 32-bit window `hi` (MSB first): len | size << 5 | advance << 9 (see
// HjdHuffTable).  t = shared-window address of the table.  Codes longer than the first-level table take
// one more load; an unassigned code yields HJD_BAD_ENTRY (advance 127).
__device__ __forceinline__ uint32_t hjd_lookup(uint32_t t, uint32_t hi)
{
    uint32_t e = hjd_lds_u16(t + ((hi >> (32 - HJD_LUT_BITS)) << 1));
    if ((e & 31u) == 0) {
        const uint32_t idx = hjd_shr((hi >> 16) & ((1u << (16 - HJD_LUT_BITS)) - 1u), (e >> 5) & 7u);
        e = hjd_lds_u16(t + HJD_TAB_LUT2_OFF + ((e >> 8) << 2) + (idx << 1));
    }
    return e;
}

// ---- the two grids of the per-image output kernels (prefix, n_items and max_items: see kernels.cuh) ----
// Images of similar size: an (image, CTA) grid, blockIdx.y = image - img_base, blockIdx.x = CTA of that image, no look-up.
// Mixed or tiny sizes (FLAT): a 1-D grid over all items of the batch, the image of each thread found by binary search.
// The 2-D grid is sized for the largest image, so one 4096x4096 image among 4096 thumbnails would launch 2 M empty CTAs
// (2.2 ms instead of 0.6), and a 16x16 image would get a CTA with one active thread; the search costs similar-sized
// batches 4 % (a chain of dependent loads in front of every CTA), an empty CTA next to nothing.

// The image that holds item `key` of the batch: the last i with prefix[i] <= key.
__device__ __forceinline__ int hjd_image_of(const uint32_t* __restrict__ prefix, int n_images, uint32_t key)
{
    int lo = 0, hi = n_images - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (prefix[mid] <= key) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// The calling thread's image d and item of that image in either grid (CTAs of CTA_THREADS threads); false when the
// thread lies past the batch's last item (FLAT).  In the 2-D grid item may lie past its image's last item: the kernel
// checks that against the image.
template <bool FLAT, uint32_t CTA_THREADS>
__device__ __forceinline__ bool hjd_locate(const HjdImageDesc* __restrict__ imgs, const uint32_t* __restrict__ prefix,
                                           int n_images, int img_base, const HjdImageDesc*& d, uint32_t& item)
{
    if (FLAT) {
        const uint32_t key = blockIdx.x * CTA_THREADS + threadIdx.x + prefix[0];
        if (key >= prefix[n_images]) return false;
        const int i = hjd_image_of(prefix, n_images, key);
        d = imgs + i;
        item = key - prefix[i];
    } else {
        d = imgs + (blockIdx.y + img_base);
        item = blockIdx.x * CTA_THREADS + threadIdx.x;
    }
    return true;
}

// The grid choice: the (image, CTA) grid unless it would have more than 4x as many thread slots as items.  An idle slot
// is cheap (config 5 runs at 1.6x: 1.02 ms against 1.11 ms with the search), so only clearly skewed or tiny-image
// batches go flat.
static inline bool hjd_grid_per_image(uint32_t max_items, int n_images, uint32_t n_items, uint32_t cta_threads)
{
    const uint64_t cols = (max_items + cta_threads - 1) / cta_threads;
    return cols * cta_threads * (uint64_t)n_images <= (uint64_t)n_items * 4;
}

// Launches kernel(args..., prefix, n_images, img_base) in the grid hjd_grid_per_image picks: `grid` as launches of at
// most 65,535 images (the limit of gridDim.y), or `flat` once over all items.
template <typename Kernel, typename... Args>
static void hjd_launch_per_image(Kernel grid, Kernel flat, uint32_t cta_threads, const uint32_t* prefix, int n_images,
                                 uint32_t n_items, uint32_t max_items, cudaStream_t st, Args... args)
{
    if (hjd_grid_per_image(max_items, n_images, n_items, cta_threads)) {
        const unsigned gx = (max_items + cta_threads - 1) / cta_threads;
        for (int base = 0; base < n_images; base += 65535)
            grid<<<dim3(gx, min(65535, n_images - base)), cta_threads, 0, st>>>(args..., nullptr, n_images, base);
    } else {
        const unsigned g = (unsigned)(((uint64_t)n_items + cta_threads - 1) / cta_threads);
        flat<<<g, cta_threads, 0, st>>>(args..., prefix, n_images, 0);
    }
}
