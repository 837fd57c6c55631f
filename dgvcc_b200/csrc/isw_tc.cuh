// Host interface of the ISW tensor-core GEMMs (isw_gram_tc.cu, isw_sx_tc.cu) for the entry points of isw_kernels.cu.
#pragma once
#include "common.cuh"

namespace dgvcc {

// The shapes the tensor-core GEMMs tile.  TMA needs 16-byte global row strides: hw % 4 == 0 for fp32 rows, hw % 8 == 0
// for fp16 / bf16 rows.  c >= 32 because tiny channel counts waste the 128-wide tile.  The rows of S in dX = S X are c
// floats (c % 4 == 0); the half Gram keeps that rule too, so a half forward and its backward accept the same shapes.
inline bool gram_tc_tiles(int c, int hw) { return hw % 4 == 0 && c >= 32; }               // fp32 Gram
inline bool sx_tc_tiles(int c, int hw) { return hw % 4 == 0 && c % 4 == 0 && c >= 32; }   // fp32 dX = S X
inline bool half_tc_tiles(int c, int hw) { return hw % 8 == 0 && c % 4 == 0 && c >= 32; } // fp16 / bf16, both GEMMs
// TMA also needs 16-byte aligned bases
inline bool tma_aligned(const void* a, const void* b = nullptr, const void* c = nullptr) {
    return !(((uintptr_t)a | (uintptr_t)b | (uintptr_t)c) & 15u);
}

namespace isw_tc {
// Split-K Gram partials of x [batch, c, hw], for isw_cov_finish_kernel.  T = float, __half or __nv_bfloat16; STD (half
// only): the partials of the standardised map  (x - mean) / sd  (* mask), the same bits as the fp32 kernel on that map.
// mean, sd [batch * c]; mask [batch, hw] or NULL.  DGVCC_ERR_UNSUPPORTED for shapes the kernel does not tile.
template <typename T, bool STD = false>
int launch(const T* x, const float* mean, const float* sd, const float* mask, int batch, int c, int hw, int splits,
           int k_per_split, float* part, cudaStream_t stream);
}  // namespace isw_tc

namespace isw_sx {
// dX_b = scale_b * (S_b X_b) with S fp32 and X, dX of type T; exact selects the variant for a TF32-exact S.  STD (half
// only, never exact): dY = S Y in fp32 with Y = (X - mean) / sd (* mask) standardised on load, the same bits as the fp32
// kernel on Y.  scale [batch] or NULL.  DGVCC_ERR_UNSUPPORTED for shapes the kernel does not tile.
template <typename T, bool STD = false>
int launch(const float* s, const T* x, const float* mean, const float* sd, const float* mask, int batch, int c, int hw,
           void* dx, const float* scale, bool exact, cudaStream_t stream);
}  // namespace isw_sx

}  // namespace dgvcc
