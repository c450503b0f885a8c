// Pillow-exact bilinear resize of uint8 RGB frames fused into the patch gather (see resize.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lwdetr_b200.h"

namespace lwb {

// frames: HOST array [B] of DEVICE frame descriptors (HWC RGB uint8; any size within the header's limits).  Each frame
// is resized to R x R as Pillow's Image.resize((R, R), BILINEAR) does, normalised as (x/255 - mean[c]) / std[c] and
// written to A [B*(R/16)^2, 768] (16-bit, window-major rows, k = c*256 + py*16 + px) - the layout of patch_gather_u8.
// Returns 0, a CUDA error code, or -2 for arguments outside the limits (the C ABI checks them first).
int resize_patch_gather_u8_launch(int dtype, const lwdetr_frame* frames, int B, int R, const float* mean, const float* stdv,
                                  void* A, cudaStream_t st);

}  // namespace lwb
