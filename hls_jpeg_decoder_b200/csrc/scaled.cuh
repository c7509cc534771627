// csrc/scaled.cuh -- launch wrapper of the reduced-size (DCT-domain scaled) decode kernel (scaled.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

// Upload the reduced IDCT's constants, computed on the host with libm (hjd_api.cu): cosN[p * N + k] =
// cosf(((2p+1) * k * 3.14f) / (2N)) for N = 4, 2, 1, and cc[u * 4 + v] = C(u) * C(v) for u, v < 4.
cudaError_t hjd_set_scaled_constants(const float cos4[16], const float cos2[4], const float cos1[1], const float cc[16]);

// Coefficients -> output at 1/2, 1/4 or 1/8 (shift 1, 2, 3) of the source size: one thread per MCU, a per-image output
// kernel over MCUs (mcu_prefix, n_mcus, max_mcus: see kernels.cuh).  Image i is written at imgs[i].rgb_off as
// ceil(W >> shift) x ceil(H >> shift) pixels, RGB24 with stride 3 * that width, or with gray (HJD_FLAG_GRAY_OUT) the
// luma samples alone (no chroma IDCT, no colour conversion), one byte per pixel, stride that width.
cudaError_t hjd_launch_scaled(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets, uint8_t* out,
                              const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus, uint32_t max_mcus, int shift,
                              bool gray, cudaStream_t st);
