// csrc/kernels.cuh -- launch wrappers of the sm_100a kernels (kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

#define HJD_IDCT_THREADS  128   // unfused IDCT kernel: one 8x8 block per thread
#define HJD_COLOR_THREADS 128   // unfused colour kernel: 16 pixels of one row per thread
#define HJD_MCU_THREADS   128   // per-MCU fused kernel: one MCU (all its blocks -> RGB) per thread

// Per-device function attributes (shared-memory windows); call after cudaSetDevice, once per batch handle.
cudaError_t hjd_kernels_init_device(void);

// Upload the IDCT constants (host libm values, loadjpg.cpp:96-102,120).
cudaError_t hjd_set_idct_constants(const float cos_tab[64], float cc0, float cc00);

// The tensor-core kernel's IDCT matrix as the 16 KB FP16 tile image it keeps in shared memory (host computation; see mcu_tc.cuh):
// row n of 128 (0..63: M_hi * 2^-13 of sample n = 8y+x; 64..127: M_lo), 64 FP16 per row in zig-zag order, 16-byte chunk j of
// row n stored at chunk j ^ (n & 7) (128-byte swizzle), rows in 1024-byte groups of eight.
void hjd_build_idct_matrix(const float cos_tab[64], float cc0, float cc00, uint16_t img[8192]);

// Kernel 0: RSTn marker scan -> interval_start[] (one CTA per image), images [first_image, first_image + n);
// scans longer than HJD_SCAN_SLICE_MIN are done by the n_slices slice CTAs instead (count, then number).
cudaError_t hjd_launch_marker_scan(const uint8_t* arena, const HjdImageDesc* imgs, uint32_t* interval_start,
                                   int32_t* status, int first_image, int n_images, const HjdScanSlice* slices,
                                   int n_slices, uint32_t* slice_cnt, cudaStream_t st);

// Kernel 1a: restart-interval-parallel Huffman decode -> int16 coefficients (zig-zag order).
cudaError_t hjd_launch_entropy_restart(const uint8_t* arena, const HjdImageDesc* imgs, const HjdTableSet* tsets,
                                       const uint32_t* interval_start, const HjdEntropyWork* work,
                                       const HjdEntropySeg* segs, int n_work,
                                       int max_tabs, int16_t* coef, int32_t* status, cudaStream_t st);

// Kernel 2: dequantise + de-zig-zag + IDCT -> u8 planes (bit-exact with the reference's direct form).
cudaError_t hjd_launch_idct_planes(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                                   uint8_t* planes, int n_images, uint32_t max_blocks, cudaStream_t st);

// Kernel 3: chroma upsample + YCbCr->RGB + clamp -> packed RGB24.
cudaError_t hjd_launch_color(const uint8_t* planes, const HjdImageDesc* imgs, uint8_t* rgb, int n_images,
                             uint32_t max_width, uint32_t max_height, cudaStream_t st);

// Per-image output kernels (hjd_launch_mcu_rgb, hjd_launch_luma, hjd_launch_scaled in scaled.cuh): one thread per item of
// an image (an MCU or a luma block), taking the items through three arguments:
//   prefix[i] = items of images 0..i-1 (any common offset; n_images + 1 entries);
//   n_items   = prefix[n_images] - prefix[0];
//   max_items = items of the largest image.
// Batches of similar-sized images get an (image, CTA) grid, mixed or tiny sizes a flat grid over all items
// (device_common.cuh).

// Kernels 2+3 fused per MCU (default path): one thread = one MCU, coefficients -> RGB, no plane traffic, no barriers.
// A per-image output kernel over MCUs (mcu_prefix, n_mcus, max_mcus).
// bmp: write the reference's BMP file layout (header at rgb_off + 10, bottom-up B G R rows from rgb_off + 64).
// variant: where the IDCT's fast tier runs and who re-evaluates the flagged samples; same bytes out.
#define HJD_MCU_CUDA_CORE    0   // FP32 FMA chains on the CUDA cores, every thread re-evaluates its own flagged samples (default)
#define HJD_MCU_TENSOR_CORE  1   // tcgen05.mma (mcu_tc.cuh), exact re-evaluations batched per warp
cudaError_t hjd_launch_mcu_rgb(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                               uint8_t* rgb, const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus,
                               uint32_t max_mcus, bool bmp, int variant, cudaStream_t st);

// Luma-only decode at full size (HJD_FLAG_GRAY_OUT): one thread = one luma block that holds a pixel of its image
// (ceil(W/8) x ceil(H/8) of them, row-major), the IDCT of the fused kernel, rows clipped at W and H; image i is
// written at imgs[i].rgb_off as W x H bytes, stride W.  Chroma blocks are not read.  A per-image output kernel over
// those luma blocks (luma_prefix, n_luma, max_luma).
#define HJD_LUMA_THREADS 128
cudaError_t hjd_launch_luma(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets, uint8_t* out,
                            const uint32_t* luma_prefix, int n_images, uint32_t n_luma, uint32_t max_luma, cudaStream_t st);
