// csrc/multiscan.cuh -- launch wrapper of the multi-scan entropy kernel (multiscan.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "hjd_types.h"

// Work items [0, n_work) of one dependency level: one thread per (scan, restart interval) -> coefficients of
// the scan's (component, band) positions.  starts: interval starts per scan (HjdScanDesc::start_base);
// tabs: the batch's per-scan Huffman tables (progressive AC tables in the raw-run layout).
cudaError_t hjd_launch_multiscan(const uint8_t* arena, const HjdImageDesc* imgs, const HjdScanDesc* scans,
                                 const HjdMsWork* work, int n_work, const uint32_t* starts, const HjdHuffTable* tabs,
                                 int16_t* coef, int32_t* status, cudaStream_t st);
