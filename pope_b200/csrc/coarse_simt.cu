// coarse_simt.cu -- coarse matching with fp32 FMA arithmetic (inputs fp32 or bf16).
//
// Replaces the op sequence of src/matcher/utils/coarse_matching.py:106-119 and :175-189 (reference tree):
//   einsum -> /T -> softmax(dim1) * softmax(dim2) -> > thr -> == rowmax -> == colmax
// without ever writing the L x S matrix.  Same three-sweep structure as the tcgen05 path (coarse_tc.cu):
//   sweep 1: row log-sum-exp of  S  = f0 f1^T * scale      (CTA owns 128 rows, streams all columns, online softmax)
//   sweep 2: row log-sum-exp of  S^T = f1 f0^T * scale      (= column log-sum-exp of S)
//   sweep 3: recompute S, t2 = (x - lse_r[i]) + (x - lse_c[j]) = log2 conf(i,j); cells with t2 > log2(thr) update
//            the best-candidate record of their row and column (64-bit atomicMax, rare).
// For thr > 0.15 sweep 3 is replaced by candidate lists filled during sweep 2 (see coarse_tc.cu / coarse_finalize.cu).
// This is the product path for fp32 inputs (tcgen05 has no true-fp32 MMA) and the on-device cross-check for
// the tensor-core path.  All quantities are in log2 units (x = <f0,f1> * log2(e)/(C*T)).
#include "common.cuh"

namespace pope {
namespace {

constexpr int BM = 128, BN = 128, BK = 16, NT = 256, LDS_PAD = 4;

template <typename T> struct Loader;
template <> struct Loader<float> {
  // 128 rows x 16 floats per chunk = 512 float4, two per thread
  static __device__ __forceinline__ void load(const float* __restrict__ base, int rows_total, int row0, int C, int k0,
                                              float (*dst)[BM + LDS_PAD], int tid) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      int idx = tid + u * NT;
      int row = idx >> 2, q = idx & 3;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + row < rows_total)
        v = __ldg(reinterpret_cast<const float4*>(base + size_t(row0 + row) * C + k0 + q * 4));
      dst[q * 4 + 0][row] = v.x; dst[q * 4 + 1][row] = v.y; dst[q * 4 + 2][row] = v.z; dst[q * 4 + 3][row] = v.w;
    }
  }
};
template <> struct Loader<__nv_bfloat16> {
  // 128 rows x 16 bf16 per chunk = 256 uint4, one per thread
  static __device__ __forceinline__ void load(const __nv_bfloat16* __restrict__ base, int rows_total, int row0, int C,
                                              int k0, float (*dst)[BM + LDS_PAD], int tid) {
    int row = tid >> 1, h = tid & 1;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (row0 + row < rows_total)
      v = __ldg(reinterpret_cast<const uint4*>(base + size_t(row0 + row) * C + k0 + h * 8));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      dst[h * 8 + 2 * e + 0][row] = __uint_as_float(w[e] << 16);
      dst[h * 8 + 2 * e + 1][row] = __uint_as_float(w[e] & 0xffff0000u);
    }
  }
};

// One 128x128 tile of A B^T (fp32 accumulate); thread (tx,ty) owns rows {ty*4+r, 64+ty*4+r} x cols {tx*4+c, 64+tx*4+c}.
template <typename T>
__device__ __forceinline__ void tile_gemm(const T* __restrict__ A, int LA, int row0, const T* __restrict__ B, int LB,
                                          int col0, int C, float (*As)[BM + LDS_PAD], float (*Bs)[BN + LDS_PAD],
                                          float (&acc)[8][8], int tid) {
  const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
  for (int k0 = 0; k0 < C; k0 += BK) {
    Loader<T>::load(A, LA, row0, C, k0, As, tid);
    Loader<T>::load(B, LB, col0, C, k0, Bs, tid);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ int frag_index(int t, int r) { return (r < 4) ? (t * 4 + r) : (64 + t * 4 + (r - 4)); }

// lse_out[n, row] = log2 sum_j 2^(x(row, j)),  x = <A_row, B_j> * scale_log2
// EMIT (two-sweep path, second sweep: A = f1, B = f0): every cell whose raw dot product exceeds the B row's bound
// (p_row > thr, see cand_bounds_kernel) is appended to that B row's candidate list.
template <typename T, bool EMIT>
__global__ void __launch_bounds__(NT) rowlse_simt_kernel(const T* __restrict__ A_all, const T* __restrict__ B_all,
                                                        int LA, int LB, int C, float scale_log2,
                                                        float* __restrict__ lse_out, const float* __restrict__ cbound,
                                                        int* __restrict__ cand_cnt, u64* __restrict__ cand,
                                                        int32_t* __restrict__ flags, const int32_t* __restrict__ gate) {
  if (gate && !(uint32_t(*gate) & POPE_FLAG_ROBUST_PATH)) return;      // fallback launch of the fp32 tensor-core path
  __shared__ __align__(16) float As[BK][BM + LDS_PAD];
  __shared__ __align__(16) float Bs[BK][BN + LDS_PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n = blockIdx.y, row0 = blockIdx.x * BM;
  const T* A = A_all + size_t(n) * LA * C;
  const T* B = B_all + size_t(n) * LB * C;
  float m_run[8], s_run[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) { m_run[r] = -INFINITY; s_run[r] = 0.f; }
  float acc[8][8];
  for (int col0 = 0; col0 < LB; col0 += BN) {
    tile_gemm<T>(A, LA, row0, B, LB, col0, C, As, Bs, acc, tid);
    if (EMIT) {
      const size_t bpad = size_t((LB + 31) / 32) * 32;       // bound rows are padded to a multiple of 32 with +inf
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int col = col0 + frag_index(tx, c);
        if (col >= LB) continue;
        const float bound = __ldg(cbound + size_t(n) * bpad + col);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const int row = row0 + frag_index(ty, r);
          if (acc[r][c] > bound && row < LA) {
            const size_t rr = size_t(n) * LB + col;
            const int slot = atomicAdd(cand_cnt + rr, 1);
            if (slot < kCandSlots) cand[rr * kCandSlots + slot] = (u64(__float_as_uint(acc[r][c])) << 32) | uint32_t(row);
            else atomicOr(reinterpret_cast<unsigned*>(flags), POPE_FLAG_CAND_OVERFLOW);
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      float tmax = -INFINITY;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        acc[r][c] *= scale_log2;
        if (col0 + frag_index(tx, c) < LB) tmax = fmaxf(tmax, acc[r][c]);
      }
#pragma unroll
      for (int o = 8; o >= 1; o >>= 1) tmax = fmaxf(tmax, __shfl_xor_sync(kFullMask, tmax, o));
      const float m_new = fmaxf(m_run[r], tmax);
      float s = s_run[r] * exp2f(m_run[r] - m_new);
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (col0 + frag_index(tx, c) < LB) s += exp2f(acc[r][c] - m_new);
      s_run[r] = s;
      m_run[r] = m_new;
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    float s = s_run[r];
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    const int row = row0 + frag_index(ty, r);
    if (tx == 0 && row < LA) lse_out[size_t(n) * LA + row] = m_run[r] + log2f(s);
  }
}

template <typename T>
__global__ void __launch_bounds__(NT) candidates_simt_kernel(const T* __restrict__ f0_all, const T* __restrict__ f1_all,
                                                            int L, int S, int C, float scale_log2, float log2_thr,
                                                            const float* __restrict__ lse_r,
                                                            const float* __restrict__ lse_c, u64* __restrict__ rowbest,
                                                            u64* __restrict__ colbest) {
  __shared__ __align__(16) float As[BK][BM + LDS_PAD];
  __shared__ __align__(16) float Bs[BK][BN + LDS_PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n = blockIdx.y, row0 = blockIdx.x * BM;
  const T* A = f0_all + size_t(n) * L * C;
  const T* B = f1_all + size_t(n) * S * C;
  float lr[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    int row = row0 + frag_index(ty, r);
    lr[r] = row < L ? lse_r[size_t(n) * L + row] : INFINITY;   // +inf -> t2 = -inf -> never a candidate
  }
  float acc[8][8];
  for (int col0 = 0; col0 < S; col0 += BN) {
    tile_gemm<T>(A, L, row0, B, S, col0, C, As, Bs, acc, tid);
    float lc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      int col = col0 + frag_index(tx, c);
      lc[c] = col < S ? __ldg(lse_c + size_t(n) * S + col) : INFINITY;
    }
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float x = acc[r][c] * scale_log2;
        const float t2 = (x - lr[r]) + (x - lc[c]);
        if (t2 > log2_thr) {
          const int row = row0 + frag_index(ty, r), col = col0 + frag_index(tx, c);
          atomicMax(rowbest + size_t(n) * L + row, pack_best(t2, col));
          atomicMax(colbest + size_t(n) * S + col, pack_best(t2, row));
        }
      }
  }
}

template <typename T>
cudaError_t run_typed(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st, bool gated) {
  const T* f0 = static_cast<const T*>(p.f0);
  const T* f1 = static_cast<const T*>(p.f1);
  const int32_t* gate = gated ? flags : nullptr;
  dim3 gr((p.L + BM - 1) / BM, p.n), gc((p.S + BM - 1) / BM, p.n);
  cudaError_t e;
  if (gated) {
    if (!two_sweeps_possible(p)) return cudaErrorInvalidValue;     // the gated form exists for the two-sweep scheme only
    if ((e = gated_clear_run(w.rowbest, w.zero_bytes, gate, st)) != cudaSuccess) return e;
  } else if ((e = cudaMemsetAsync(w.rowbest, 0, w.zero_bytes, st)) != cudaSuccess) {
    return e;
  }
  rowlse_simt_kernel<T, false><<<gr, NT, 0, st>>>(f0, f1, p.L, p.S, p.C, p.scale_log2, w.lse_r, nullptr, nullptr, nullptr, nullptr,
                                                  gate);
  if (two_sweeps_possible(p)) {
    // same two-sweep scheme as the tcgen05 path: the column sweep lists the cells with p_row > thr
    if ((e = cand_bounds_run(p, w, st, gate)) != cudaSuccess) return e;
    rowlse_simt_kernel<T, true><<<gc, NT, 0, st>>>(f1, f0, p.S, p.L, p.C, p.scale_log2, w.lse_c, w.cbound, w.cand_cnt, w.cand, flags,
                                                   gate);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cand_eval_run(p, w, st, gate);
  }
  rowlse_simt_kernel<T, false><<<gc, NT, 0, st>>>(f1, f0, p.S, p.L, p.C, p.scale_log2, w.lse_c, nullptr, nullptr, nullptr, nullptr,
                                                  nullptr);
  candidates_simt_kernel<T><<<gr, NT, 0, st>>>(f0, f1, p.L, p.S, p.C, p.scale_log2, p.log2_thr, w.lse_r, w.lse_c,
                                                w.rowbest, w.colbest);
  return cudaGetLastError();
}

}  // namespace

cudaError_t coarse_simt_run(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st, bool gated) {
  return p.dtype == POPE_BF16 ? run_typed<__nv_bfloat16>(p, w, flags, st, gated) : run_typed<float>(p, w, flags, st, gated);
}

}  // namespace pope
