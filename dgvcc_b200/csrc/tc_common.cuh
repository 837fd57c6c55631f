// Raw-PTX helpers shared by the tcgen05 / TMA kernels (isw_gram_tc.cu, isw_sx_tc.cu): mbarrier, TMA tensor
// loads, UMMA issue / commit, TMEM loads, TF32 rounding, and the driver entry point for tensor maps.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace dgvcc {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// tcgen05.mma kind::tf32, cta_group::1, D (fp32) in TMEM, A and B from shared-memory descriptors.
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(a), "l"(b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ float tf32_round(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}


// Shared-memory matrix descriptor, Blackwell version bits.  lbo / sbo in bytes.
// layout_type: 2 = SWIZZLE_128B (16-byte atoms); 1 = SWIZZLE_128B_BASE32B (32-byte atoms), the only
// layout the tensor core accepts for MN-major TF32 operands.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(lbo_bytes >> 4) << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;   // descriptor version (sm_100)
    d |= (uint64_t)layout_type << 61;
    return d;
}
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return umma_desc(smem_addr, lbo_bytes, sbo_bytes, 2);
}

// Instruction descriptor for kind::tf32 with fp32 accumulation.  b_mn_major: B stored with N contiguous.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int m, int n, bool b_mn_major) {
    return (1u << 4) /*D = f32*/ | (2u << 7) /*A = tf32*/ | (2u << 10) /*B = tf32*/ |
           ((b_mn_major ? 1u : 0u) << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// cuTensorMapEncodeTiled through the runtime, so the library does not link libcuda (it must load on
// machines without a driver: the host-only checks of tests/test_abi.py).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 3-D tensor map {inner, rows, batch} of elem_bytes-wide elements with a {box_inner, box_rows, box_batch} box.
inline bool make_tmap_3d(CUtensorMap* map, CUtensorMapDataType type, uint32_t elem_bytes, const void* base, uint64_t inner,
                         uint64_t rows, uint64_t batch, uint32_t box_inner, uint32_t box_rows, CUtensorMapSwizzle swizzle,
                         uint32_t box_batch) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t dims[3] = {inner, rows, batch};
    const cuuint64_t strides[2] = {inner * elem_bytes, inner * rows * elem_bytes};
    const cuuint32_t box[3] = {box_inner, box_rows, box_batch};
    const cuuint32_t estr[3] = {1, 1, 1};
    return enc(map, type, 3, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// fp32 3-D tensor map {inner, rows, batch} with a {32 floats (one 128-byte swizzle row), box_rows, box_batch} box.
inline bool make_tmap_f32_3d(CUtensorMap* map, const float* base, uint64_t inner, uint64_t rows, uint64_t batch,
                             uint32_t box_rows, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B,
                             uint32_t box_batch = 1) {
    return make_tmap_3d(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, inner, rows, batch, 32, box_rows, swizzle, box_batch);
}

// Half-precision input (fp16 / bf16) of the ISW tensor-core kernels.  Every finite value widens to fp32 exactly, with
// zero low 13 mantissa bits: it IS its own TF32 hi part, and the lo part of the 3xTF32 split is exactly 0.
template <typename T> struct HalfIn;
template <> struct HalfIn<__half> {
    static constexpr CUtensorMapDataType TMA = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    static __device__ __forceinline__ float widen(__half v) { return __half2float(v); }
    static __device__ __forceinline__ __half narrow(float v) { return __float2half_rn(v); }
};
template <> struct HalfIn<__nv_bfloat16> {
    static constexpr CUtensorMapDataType TMA = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    static __device__ __forceinline__ float widen(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ __nv_bfloat16 narrow(float v) { return __float2bfloat16_rn(v); }
};

// four consecutive half-precision elements (8 bytes) widened to a float4
template <typename T>
__device__ __forceinline__ float4 widen4(const T* p) {
    const uint2 raw = *reinterpret_cast<const uint2*>(p);
    const T* h = reinterpret_cast<const T*>(&raw);
    return make_float4(HalfIn<T>::widen(h[0]), HalfIn<T>::widen(h[1]), HalfIn<T>::widen(h[2]), HalfIn<T>::widen(h[3]));
}

// four fp32 values rounded to nearest into four consecutive half-precision elements (one 8-byte store)
template <typename T>
__device__ __forceinline__ void narrow4(T* p, float a, float b, float c, float d) {
    T h[4] = {HalfIn<T>::narrow(a), HalfIn<T>::narrow(b), HalfIn<T>::narrow(c), HalfIn<T>::narrow(d)};
    *reinterpret_cast<uint2*>(p) = *reinterpret_cast<const uint2*>(h);
}

}  // namespace tc
}  // namespace dgvcc
