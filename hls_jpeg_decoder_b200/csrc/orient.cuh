// csrc/orient.cuh -- launch wrapper of the EXIF orientation pass (orient.cu, HJD_FLAG_EXIF_ORIENT).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

#define HJD_ORIENT_THREADS 256

// Writes every job's staged w x h image (bpp 3 or 1 bytes per pixel, rows top-down, stride w * bpp, at out + src_off)
// turned by its orientation at out + dst_off (stride out_w * bpp).  One CTA per output tile of HJD_ORIENT_TILE^2 pixels
// (batch_plan.h); tile_prefix[k] = tiles of jobs 0..k-1 (any common offset; n_jobs + 1 entries), n_tiles =
// tile_prefix[n_jobs] - tile_prefix[0].  Source and destination regions must not overlap.
cudaError_t hjd_launch_orient(uint8_t* out, const HjdOrientJob* jobs, const uint32_t* tile_prefix, int n_jobs,
                              uint32_t n_tiles, int bpp, cudaStream_t st);
