// csrc/scaled.cuh -- launch wrapper of the reduced-size (DCT-domain scaled) decode kernel (scaled.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

// Upload the reduced IDCT's constants, computed on the host with libm (hjd_api.cu): cosN[p * N + k] =
// cosf(((2p+1) * k * 3.14f) / (2N)) for N = 4, 2, 1, and cc[u * 4 + v] = C(u) * C(v) for u, v < 4.
cudaError_t hjd_set_scaled_constants(const float cos4[16], const float cos2[4], const float cos1[1], const float cc[16]);

// Coefficients -> RGB at 1/2, 1/4 or 1/8 (shift 1, 2, 3) of the source size: one thread per MCU, the grids of
// hjd_launch_mcu_rgb (mcu_prefix, n_mcus and max_mcus mean the same).  Image i is written at imgs[i].rgb_off as
// ceil(W >> shift) x ceil(H >> shift) RGB24, stride 3 * that width.
cudaError_t hjd_launch_mcu_rgb_scaled(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                                      uint8_t* rgb, const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus,
                                      uint32_t max_mcus, int shift, cudaStream_t st);
// The same for HJD_FLAG_GRAY_OUT: the luma samples only (no chroma IDCT, no colour conversion), written at imgs[i].rgb_off
// as ceil(W >> shift) x ceil(H >> shift) bytes, stride that width.
cudaError_t hjd_launch_luma_scaled(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                                   uint8_t* out, const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus,
                                   uint32_t max_mcus, int shift, cudaStream_t st);
