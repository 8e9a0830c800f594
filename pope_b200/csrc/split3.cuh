// split3.cuh -- fp32 -> three bf16 planes, a = a1 + a2 + a3, for the fp32-accuracy tcgen05 paths (the coarse sweep's MODE 4
// in coarse_tc.cu, the fp32 coarse transformer in coarse_tf.cu).  Each plane carries 8 mantissa bits and every residual
// is exact in fp32, so for normal values down to 2^-110 the three planes hold the fp32 value exactly; below that the third
// plane runs into the bf16 subnormal range and the split is exact to within 2^-134.  A contraction keeps the six
// significant products a1b1 + a2b1 + a3b1 + a1b2 + a2b2 + a1b3; the dropped ones are below 2^-24 of |a||b|.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace pope {
namespace {   // (a kernel defined in a header: one private copy per translation unit)

__device__ __forceinline__ void split3_range(const float4* __restrict__ in, uint2* __restrict__ p1, uint2* __restrict__ p2,
                                             uint2* __restrict__ p3, size_t n4) {
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += size_t(gridDim.x) * blockDim.x) {
    const float4 a = __ldcs(in + i);
    const float v[4] = {a.x, a.y, a.z, a.w};
    uint32_t h1[4], h2[4], h3[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __nv_bfloat16 b1 = __float2bfloat16_rn(v[e]);
      const float r1 = v[e] - __bfloat162float(b1);
      const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
      const float r2 = r1 - __bfloat162float(b2);
      const __nv_bfloat16 b3 = __float2bfloat16_rn(r2);
      h1[e] = __bfloat16_as_ushort(b1); h2[e] = __bfloat16_as_ushort(b2); h3[e] = __bfloat16_as_ushort(b3);
    }
    p1[i] = make_uint2(h1[0] | (h1[1] << 16), h1[2] | (h1[3] << 16));
    p2[i] = make_uint2(h2[0] | (h2[1] << 16), h2[2] | (h2[3] << 16));
    p3[i] = make_uint2(h3[0] | (h3[1] << 16), h3[2] | (h3[3] << 16));
  }
}

__global__ void __launch_bounds__(256) split3_kernel(const float4* __restrict__ in, uint2* __restrict__ p1, uint2* __restrict__ p2,
                                                    uint2* __restrict__ p3, size_t n4) {
  split3_range(in, p1, p2, p3, n4);
}

// fp32 [elems] -> three bf16 planes `stride` bytes apart (elems a multiple of 4, src 16-byte aligned)
inline cudaError_t split_planes(const float* src, __nv_bfloat16* dst, size_t stride, size_t elems, cudaStream_t st) {
  char* d = reinterpret_cast<char*>(dst);
  split3_kernel<<<148 * 8, 256, 0, st>>>(reinterpret_cast<const float4*>(src), reinterpret_cast<uint2*>(d),
                                         reinterpret_cast<uint2*>(d + stride), reinterpret_cast<uint2*>(d + 2 * stride),
                                         elems / 4);
  return cudaGetLastError();
}

}  // namespace
}  // namespace pope
