// coarse_tf.cu -- the coarse-level LoFTR transformer (d_model 256, 8 heads, linear attention) in bf16 on sm_100a, and the
// position-encoding / token-major layout step in front of it.
//
// Replaces, for bf16 coarse features, the op sequence of the reference's
//   src/matcher/matcher.py:57-58                        (pos_encoding + rearrange 'n c h w -> n (h w) c')
//   src/matcher/loftr_module/transformer.py:34-58      (LoFTREncoderLayer.forward at d_model 256)
//   src/matcher/loftr_module/linear_attention.py:21-47 (elu(x)+1 feature map, KV = K^T V / S, Z = 1/(Q . sum K + eps))
//   src/matcher/loftr_module/transformer.py:95-104     ('self' / 'cross' layer schedule)
// Every Linear is one launch of coarse_gemm_kernel: a persistent tcgen05 GEMM over items of 128 token rows x 256 output
// columns whose A (activations) and B (weights) tiles both stream through a TMA ring (the MLP weights, 512 KB and
// 256 KB, do not fit in shared memory; the q/k/v/merge weights are re-read from L2), with the accumulator of an item in
// TMEM and an epilogue that applies what follows the Linear in the reference (feature map, 1/S scale, ReLU, LayerNorm
// over the 256 channels of a row, residual) before the row leaves as bf16.  The attention is global over each pair's
// source tokens: KV^T and sum k per (pair, head) are reduced over token chunks, the chunk partials summed in a fixed
// order (no float atomics: results are bit-reproducible and a pair's output does not depend on its batch neighbours),
// then applied per token.  Activations are bf16 in HBM, all arithmetic accumulates in fp32.
#include <cuda.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace pope {
namespace {

using namespace tc1;

constexpr int kC = 256;                          // coarse d_model
constexpr int kHeads = 8, kHeadDim = 32;
constexpr int kTile = 128;                       // token rows per item (MMA M)
constexpr int kNTile = 256;                      // output columns per item (MMA N; one TMEM accumulator of 256 columns)
constexpr int kBoxK = 64;                        // bf16 elements per 128-byte swizzle row
constexpr int kABytes = kTile * kBoxK * 2;       // 16 KB activation box
constexpr int kWBytes = kNTile * kBoxK * 2;      // 32 KB weight box
constexpr int kStageBytes = kABytes + kWBytes;
constexpr int kStages = 4;
constexpr int kEpiWarps = 8;                     // two sets of four (one warp per TMEM lane quadrant); sets alternate items
constexpr int kThreads = 64 + kEpiWarps * 32;    // warp 0: TMA, warp 1: TMEM allocator + MMA, warps 2-9: epilogue
constexpr int kStageOutBytes = 32 * 128;         // per epilogue warp: 32 rows x 64 bf16 columns, 128B-swizzled
// layout: [staging: 8 x 4 KB][barriers][ring: stages x (A 16 KB + W 32 KB)], plus 1 KB alignment slack
constexpr int kSmemOut = 0;
constexpr int kSmemBar = kEpiWarps * kStageOutBytes;
constexpr int kNumBars = 2 * kStages + 4 + kEpiWarps;
constexpr int kSmemTmemPtr = kSmemBar + kNumBars * 8;
constexpr int kSmemRing = kSmemBar + 1024;
static_assert(kSmemTmemPtr + 16 <= kSmemRing, "barrier block overlaps the ring");
constexpr int kSmemAlloc = kSmemRing + kStages * kStageBytes + 1024;
static_assert(kSmemAlloc <= 227 * 1024, "coarse GEMM shared memory");

// what follows the Linear in the reference, applied to the fp32 accumulator row
enum EpiMode : int { EPI_ELU1 = 0, EPI_SCALE = 1, EPI_RELU = 2, EPI_LN = 3, EPI_LN_RES = 4 };

struct GemmParams {
  int T;                 // token rows
  int kchunks;           // K / 64
  int ksplit;            // k-chunks [0, ksplit) come from mapA0, the rest from mapA1 (torch.cat along the channels)
  int ntn;               // N / 256 (<= 3); output block j of every row tile goes through mapO<j>
  int mode[3];
  float scale;           // EPI_SCALE
  const float* gamma;    // EPI_LN / EPI_LN_RES: [256]
  const float* beta;
};

__global__ void __launch_bounds__(kThreads, 1)
coarse_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                   const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapO0,
                   const __grid_constant__ CUtensorMap mapO1, const __grid_constant__ CUtensorMap mapO2,
                   const __grid_constant__ CUtensorMap mapR, const GemmParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_full = sbase + kSmemBar, bar_empty = bar_full + 8 * kStages;
  const uint32_t bar_acc_full = bar_empty + 8 * kStages, bar_acc_empty = bar_acc_full + 16;
  const uint32_t bar_res = bar_acc_empty + 16;   // one per epilogue warp
  const uint32_t ring = sbase + kSmemRing;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kSmemTmemPtr);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (P.T + kTile - 1) / kTile, nitems = ntiles * P.ntn;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA0); prefetch_tmap(&mapA1); prefetch_tmap(&mapW);
    prefetch_tmap(&mapO0); prefetch_tmap(&mapO1); prefetch_tmap(&mapO2); prefetch_tmap(&mapR);
    for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(bar_acc_full + 8 * s, 1); mbar_init(bar_acc_empty + 8 * s, 4); }
    for (int s = 0; s < kEpiWarps; ++s) mbar_init(bar_res + 8 * s, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(sbase + kSmemTmemPtr, 512u);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
        const int t = it / P.ntn, j = it - t * P.ntn;
        for (int kc = 0; kc < P.kchunks; ++kc) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1);
          const uint32_t dst = ring + stage * kStageBytes;
          mbar_expect_tx(bar_full + 8 * stage, kStageBytes);
          if (kc < P.ksplit) tma_load_2d(dst, &mapA0, bar_full + 8 * stage, kc * kBoxK, t * kTile);
          else tma_load_2d(dst, &mapA1, bar_full + 8 * stage, (kc - P.ksplit) * kBoxK, t * kTile);
          tma_load_2d(dst + kABytes, &mapW, bar_full + 8 * stage, kc * kBoxK, j * kNTile);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16(kTile, kNTile);
      int stage = 0;
      uint32_t phase = 0, li = 0;
      for (int it = blockIdx.x; it < nitems; it += gridDim.x, ++li) {
        const uint32_t slot = li & 1;
        mbar_wait(bar_acc_empty + 8 * slot, ((li >> 1) & 1) ^ 1);      // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + slot * kNTile;
        for (int kc = 0; kc < P.kchunks; ++kc) {
          mbar_wait(bar_full + 8 * stage, phase);
          tc_fence_after();
          const uint32_t a_addr = ring + stage * kStageBytes, b_addr = a_addr + kABytes;
#pragma unroll
          for (int ks = 0; ks < kBoxK / 16; ++ks)
            umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), idesc, (kc | ks) ? 1u : 0u);
          umma_commit(bar_empty + 8 * stage);                           // ring slot free once these MMAs have read it
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(bar_acc_full + 8 * slot);
      }
    }
  } else {
    // =============================== epilogue: thread = token row, 256 channels in two passes of 128 ================
    const int ew = warp - 2, set = ew >> 2, quad = warp & 3;
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    const uint32_t stage_buf = sbase + kSmemOut + ew * kStageOutBytes;
    const uint32_t my_row = stage_buf + lane * 128;
    const uint32_t sw = uint32_t(lane & 7);
    const uint32_t bar_my_res = bar_res + 8 * ew;
    uint32_t res_phase = 0, li = 0;
    for (int it = blockIdx.x; it < nitems; it += gridDim.x, ++li) {
      if ((li & 1u) != uint32_t(set)) continue;
      const uint32_t slot = li & 1;
      const int t = it / P.ntn, j = it - t * P.ntn;
      const int mode = j == 0 ? P.mode[0] : (j == 1 ? P.mode[1] : P.mode[2]);   // (no dynamic index: P stays in param space)
      const int row0 = t * kTile + quad * 32;
      const CUtensorMap* mo = j == 0 ? &mapO0 : (j == 1 ? &mapO1 : &mapO2);
      const uint32_t taddr = tmem_base + lane_addr + slot * kNTile;
      mbar_wait(bar_acc_full + 8 * slot, (li >> 1) & 1);
      tc_fence_after();
      float mean = 0.f, rstd = 0.f;
      if (mode >= EPI_LN) {            // nn.LayerNorm statistics over both 128-column halves: mean first, then variance (64 columns per pass)
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 1
        for (int qc = 0; qc < 4; ++qc) {
          float v[64];
          tmem_ld32(taddr + qc * 64, v);
          tmem_ld32(taddr + qc * 64 + 32, v + 32);
#pragma unroll
          for (int c = 0; c < 64; c += 4) { s0 += v[c]; s1 += v[c + 1]; s2 += v[c + 2]; s3 += v[c + 3]; }
        }
        mean = ((s0 + s1) + (s2 + s3)) * (1.f / kC);
        s0 = s1 = s2 = s3 = 0.f;
#pragma unroll 1
        for (int qc = 0; qc < 4; ++qc) {
          float v[64];
          tmem_ld32(taddr + qc * 64, v);
          tmem_ld32(taddr + qc * 64 + 32, v + 32);
#pragma unroll
          for (int c = 0; c < 64; c += 4) {
            const float d0 = v[c] - mean, d1 = v[c + 1] - mean, d2 = v[c + 2] - mean, d3 = v[c + 3] - mean;
            s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
          }
        }
        rstd = rsqrtf(((s0 + s1) + (s2 + s3)) * (1.f / kC) + 1e-5f);      // biased variance, eps 1e-5
      }
#pragma unroll 1
      for (int qc = 0; qc < 4; ++qc) {   // 64 columns per pass: one staging box, 64 live values (no spills at 168 regs)
        const int col = qc * 64;
        float v[64];
        tmem_ld32(taddr + col, v);
        tmem_ld32(taddr + col + 32, v + 32);
        if (qc == 3) {                 // last read of this accumulator
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_acc_empty + 8 * slot);
        }
        if (mode == EPI_ELU1) {
#pragma unroll
          for (int c = 0; c < 64; ++c) v[c] = v[c] > 0.f ? v[c] + 1.f : ex2_approx(v[c] * kLog2e);
        } else if (mode == EPI_SCALE) {
#pragma unroll
          for (int c = 0; c < 64; ++c) v[c] *= P.scale;
        } else if (mode == EPI_RELU) {
#pragma unroll
          for (int c = 0; c < 64; ++c) v[c] = fmaxf(v[c], 0.f);
        } else {
          const float4* g4 = reinterpret_cast<const float4*>(P.gamma + col);
          const float4* b4 = reinterpret_cast<const float4*>(P.beta + col);
#pragma unroll
          for (int c = 0; c < 64; c += 4) {
            const float4 g = __ldg(g4 + (c >> 2)), b = __ldg(b4 + (c >> 2));
            v[c] = fmaf((v[c] - mean) * rstd, g.x, b.x); v[c + 1] = fmaf((v[c + 1] - mean) * rstd, g.y, b.y);
            v[c + 2] = fmaf((v[c + 2] - mean) * rstd, g.z, b.z); v[c + 3] = fmaf((v[c + 3] - mean) * rstd, g.w, b.w);
          }
        }
        if (lane == 0) tma_store_wait_read();                   // the previous store out of this box has read it
        __syncwarp();
        if (mode == EPI_LN_RES) {                                // + x: the residual rows through the staging box
          if (lane == 0) {
            mbar_expect_tx(bar_my_res, kStageOutBytes);
            tma_load_2d(stage_buf, &mapR, bar_my_res, col, row0);
          }
          __syncwarp();
          mbar_wait(bar_my_res, res_phase);
          res_phase ^= 1;
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) {
            uint4 r;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                         : "r"(my_row + ((uint32_t(c8) ^ sw) << 4)));
            const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[c8 * 8 + 2 * e] += __uint_as_float(w[e] << 16);
              v[c8 * 8 + 2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
            }
          }
          __syncwarp();
        }
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          const int c = c8 * 8;
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                       ::"r"(my_row + ((uint32_t(c8) ^ sw) << 4)), "r"(pack_bf16(v[c], v[c + 1])),
                         "r"(pack_bf16(v[c + 2], v[c + 3])), "r"(pack_bf16(v[c + 4], v[c + 5])),
                         "r"(pack_bf16(v[c + 6], v[c + 7])) : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(mo, stage_buf, col, row0);              // rows past T are clipped by the tensor map
          tma_store_commit();
        }
      }
    }
    if (lane == 0) tma_store_wait_all();                        // global writes complete before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512u);
  }
}

// ---- global linear attention ----------------------------------------------------------------------------------------
// k already holds elu(.)+1 and v holds values / S (fused into the projection's epilogue).  Per pair and head h:
//   KV[d][e] = sum_s k[s][d] v[s][e],  ksum[d] = sum_s k[s][d],  msg[l][e] = S * (q[l] . KV[:, e]) / (q[l] . ksum + eps)
// The reduction over s runs in chunks of kKvChunk tokens (one block per (chunk, pair), warp = head, lane = d); a second
// kernel sums the chunk partials in chunk order.  Chunks never straddle pairs.
constexpr int kKvChunk = 128;
constexpr int kKvRows = kHeadDim + 1;                   // 32 rows of KV and the row of sum_s k
constexpr int kKvFloats = kHeads * kKvRows * kHeadDim;  // per pair (or per chunk partial)
constexpr int kApplyTokens = 128;

__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// part[((b * nch + c) * kHeads + h) * kKvRows + e) * 32 + d]: e < 32 -> KV[d][e] over the chunk, e == 32 -> sum k[d]
__global__ void __launch_bounds__(kHeads * 32)
coarse_kv_partial_kernel(const __nv_bfloat16* __restrict__ k, const __nv_bfloat16* __restrict__ v, int S, int nch,
                         float* __restrict__ part) {
  const int c = blockIdx.x, b = blockIdx.y, h = threadIdx.x >> 5, d = threadIdx.x & 31;
  const int s0 = c * kKvChunk, s1 = min(S, s0 + kKvChunk);
  float acc[kHeadDim], ks = 0.f;
#pragma unroll
  for (int e = 0; e < kHeadDim; ++e) acc[e] = 0.f;
  const __nv_bfloat16* kp = k + (size_t(b) * S + s0) * kC + h * kHeadDim + d;
  const uint4* vp = reinterpret_cast<const uint4*>(v + (size_t(b) * S + s0) * kC + h * kHeadDim);
#pragma unroll 4
  for (int s = s0; s < s1; ++s, kp += kC, vp += kC / 8) {
    const float kd = __bfloat162float(*kp);
    uint4 q4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) q4[i] = __ldg(vp + i);             // the same 64 bytes in every lane: one broadcast
    const uint32_t w[16] = {q4[0].x, q4[0].y, q4[0].z, q4[0].w, q4[1].x, q4[1].y, q4[1].z, q4[1].w,
                            q4[2].x, q4[2].y, q4[2].z, q4[2].w, q4[3].x, q4[3].y, q4[3].z, q4[3].w};
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      acc[2 * i] = fmaf(kd, bf_lo(w[i]), acc[2 * i]);
      acc[2 * i + 1] = fmaf(kd, bf_hi(w[i]), acc[2 * i + 1]);
    }
    ks += kd;
  }
  float* out = part + ((size_t(b) * nch + c) * kHeads + h) * kKvRows * kHeadDim + d;
#pragma unroll
  for (int e = 0; e < kHeadDim; ++e) out[e * kHeadDim] = acc[e];
  out[kHeadDim * kHeadDim] = ks;
}

// kv[((b * kHeads + h) * kKvRows + r) * 32 + x]: r < 32 -> KV[d = r][e = x], r == 32 -> sum k[d = x]; chunks in order
__global__ void __launch_bounds__(kHeads * 32)
coarse_kv_reduce_kernel(const float* __restrict__ part, int nch, float* __restrict__ kv) {
  const int b = blockIdx.x, h = threadIdx.x >> 5, d = threadIdx.x & 31;
  const float* src = part + (size_t(b) * nch * kHeads + h) * kKvRows * kHeadDim + d;
  float* dst = kv + (size_t(b) * kHeads + h) * kKvRows * kHeadDim;
  for (int e = 0; e < kKvRows; ++e) {
    float s = 0.f;
    for (int c = 0; c < nch; ++c) s += src[size_t(c) * kKvFloats + e * kHeadDim];
    if (e < kHeadDim) dst[d * kHeadDim + e] = s;
    else dst[kHeadDim * kHeadDim + d] = s;
  }
}

// one block per (kApplyTokens tokens, pair); warp = head, lane = output column e of the head
__global__ void __launch_bounds__(kHeads * 32)
coarse_attn_apply_kernel(const __nv_bfloat16* __restrict__ q, const float* __restrict__ kv, int L, int S, float eps,
                         __nv_bfloat16* __restrict__ msg) {
  const int b = blockIdx.y, h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* kvh = kv + (size_t(b) * kHeads + h) * kKvRows * kHeadDim;
  float kvc[kHeadDim], ksum[kHeadDim];
#pragma unroll
  for (int d = 0; d < kHeadDim; ++d) {
    kvc[d] = kvh[d * kHeadDim + lane];
    ksum[d] = kvh[kHeadDim * kHeadDim + d];
  }
  const float fs = float(S);
  const int l0 = blockIdx.x * kApplyTokens, l1 = min(L, l0 + kApplyTokens);
  for (int l = l0; l < l1; ++l) {
    const size_t off = (size_t(b) * L + l) * kC + h * kHeadDim + lane;
    const float ql = __bfloat162float(q[off]);
    float o = 0.f, z = 0.f;
#pragma unroll
    for (int d = 0; d < kHeadDim; ++d) {
      const float qd = __shfl_sync(kFullMask, ql, d);
      o = fmaf(qd, kvc[d], o);
      z = fmaf(qd, ksum[d], z);
    }
    msg[off] = __float2bfloat16_rn(o * fs / (z + eps));
  }
}

// ---- position encoding + layout: out[b, y W + x, c] = bf16(feat[b, c, y, x] + pe[c, y, x]) ---------------------------
constexpr int kPePix = 32;

__global__ void __launch_bounds__(256)
coarse_pos_encode_kernel(const float* __restrict__ feat, const float* __restrict__ pe, int H, int W, int pe_h, int pe_w,
                         __nv_bfloat16* __restrict__ out) {
  __shared__ float tile[kPePix][kC + 1];
  const int b = blockIdx.y, p0 = blockIdx.x * kPePix, HW = H * W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int p = p0 + lane;
  if (p < HW) {                                      // read: lane = pixel (coalesced along x), warps stride the channels
    const int y = p / W, x = p - y * W;
    for (int c = warp; c < kC; c += 8)
      tile[lane][c] = feat[(size_t(b) * kC + c) * HW + p] + pe[(size_t(c) * pe_h + y) * pe_w + x];
  }
  __syncthreads();
  for (int pp = warp; pp < kPePix && p0 + pp < HW; pp += 8) {   // write: lane = 8 channels of one token row
    const float* r = &tile[pp][lane * 8];
    *reinterpret_cast<uint4*>(out + (size_t(b) * HW + p0 + pp) * kC + lane * 8) =
        make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct Dst { void* ptr; int64_t pitch; };         // one 256-column output block (bf16, row pitch in elements)

// Y[T, N] = epilogue(cat(A0[T, K0], A1[T, K1]) . W[N, K0 + K1]^T); out[j] receives output columns [256 j, 256 j + 256).
// resid (EPI_LN_RES): [T, 256] rows added after the LayerNorm.
cudaError_t gemm_run(int64_t T, const void* A0, int K0, const void* A1, int K1, const void* W, int N, const Dst (&out)[3],
                     GemmParams P, const void* resid, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  const int K = K0 + K1;
  if (T > 0x7fffffff - kTile || N % kNTile || N / kNTile > 3 || K0 % kBoxK || K1 % kBoxK) return cudaErrorInvalidValue;
  CUtensorMap ma0, ma1, mw, mo[3], mr;
  if (!make_map2d(&ma0, A0, T, K0, K0)) return cudaErrorInvalidValue;
  if (!make_map2d(&ma1, K1 ? A1 : A0, T, K1 ? K1 : K0, K1 ? K1 : K0)) return cudaErrorInvalidValue;
  if (!make_map2d(&mw, W, N, K, K, kNTile)) return cudaErrorInvalidValue;
  for (int j = 0; j < 3; ++j) {
    const Dst& o = out[j < N / kNTile ? j : 0];   // unused maps still have to be valid descriptors
    if (!o.ptr || !make_map2d(&mo[j], o.ptr, T, kNTile, o.pitch, 32)) return cudaErrorInvalidValue;
  }
  if (!make_map2d(&mr, resid ? resid : out[0].ptr, T, kC, resid ? kC : out[0].pitch, 32)) return cudaErrorInvalidValue;
  P.T = int(T);
  P.kchunks = K / kBoxK;
  P.ksplit = K0 / kBoxK;
  P.ntn = N / kNTile;
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(coarse_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemAlloc)) != cudaSuccess)
    return e;
  const int64_t nitems = (T + kTile - 1) / kTile * P.ntn;
  coarse_gemm_kernel<<<unsigned(nitems < sms ? nitems : sms), kThreads, kSmemAlloc, st>>>(ma0, ma1, mw, mo[0], mo[1], mo[2],
                                                                                         mr, P);
  return cudaGetLastError();
}

// packed weights of one d_model-256 LoFTREncoderLayer (byte offsets; matrices bf16 row-major [out, in] like nn.Linear)
constexpr size_t kOffQkv = 0;                                  // [768, 256]  q_proj, k_proj, v_proj stacked
constexpr size_t kOffMerge = kOffQkv + 768 * 256 * 2;          // [256, 256]
constexpr size_t kOffMlp1 = kOffMerge + 256 * 256 * 2;         // [512, 512]
constexpr size_t kOffMlp2 = kOffMlp1 + 512 * 512 * 2;          // [256, 512]
constexpr size_t kOffLn = kOffMlp2 + 256 * 512 * 2;            // fp32: norm1.weight, norm1.bias, norm2.weight, norm2.bias
constexpr size_t kLayerBytes = kOffLn + 4 * 256 * 4;
static_assert(kLayerBytes == POPE_COARSE_TF_LAYER_BYTES, "include/pope_b200.h documents this layout");

// five [n * max(L, S), 256] bf16 planes (q, k, v, msg, m1; the MLP's hidden [T, 512] spans the q and k planes, which are
// dead by then), the per-chunk KV partials and the reduced KV of every pair
struct CoarseTfScratch { __nv_bfloat16 *q, *k, *v, *msg, *m1, *hid; float *part, *kv; int nch; size_t bytes; };
CoarseTfScratch carve_coarse_tf(void* base, int64_t n, int L, int S) {
  CoarseTfScratch w;
  char* p = static_cast<char*>(base);
  const int lmax = L > S ? L : S;
  const size_t unit = align_up(size_t(n) * lmax * kC * 2, 256);
  w.nch = (lmax + kKvChunk - 1) / kKvChunk;
  size_t off = 0;
  w.q = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.k = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.v = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.msg = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.m1 = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.hid = w.q;
  w.part = reinterpret_cast<float*>(p + off); off += align_up(size_t(n) * w.nch * kKvFloats * 4, 256);
  w.kv = reinterpret_cast<float*>(p + off); off += align_up(size_t(n) * kKvFloats * 4, 256);
  w.bytes = off;
  return w;
}

// x <- x + norm2(mlp(cat(x, norm1(merge(attention(q(x), k(src), v(src)))))))      (transformer.py:34-58), in place on x
// x: [n, Lx, 256], src: [n, Ls, 256]
cudaError_t encoder_layer(__nv_bfloat16* x, const __nv_bfloat16* src, int64_t n, int Lx, int Ls, const char* wl,
                          const CoarseTfScratch& w, cudaStream_t st) {
  const int64_t Tx = n * Lx, Ts = n * Ls;
  const float* ln = reinterpret_cast<const float*>(wl + kOffLn);
  const Dst none{nullptr, 0};
  cudaError_t e;
  GemmParams P{};
  if (x == src) {                       // self: one pass over x produces q, k, v
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_ELU1; P.mode[2] = EPI_SCALE; P.scale = 1.f / float(Ls);
    const Dst o[3] = {{w.q, kC}, {w.k, kC}, {w.v, kC}};
    if ((e = gemm_run(Tx, x, kC, nullptr, 0, wl + kOffQkv, 768, o, P, nullptr, st)) != cudaSuccess) return e;
  } else {
    P.mode[0] = EPI_ELU1;
    const Dst oq[3] = {{w.q, kC}, none, none};
    if ((e = gemm_run(Tx, x, kC, nullptr, 0, wl + kOffQkv, 256, oq, P, nullptr, st)) != cudaSuccess) return e;
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_SCALE; P.scale = 1.f / float(Ls);
    const Dst okv[3] = {{w.k, kC}, {w.v, kC}, none};
    if ((e = gemm_run(Ts, src, kC, nullptr, 0, wl + kOffQkv + 256 * 256 * 2, 512, okv, P, nullptr, st)) != cudaSuccess)
      return e;
  }
  const int nch = (Ls + kKvChunk - 1) / kKvChunk;
  coarse_kv_partial_kernel<<<dim3(nch, unsigned(n)), kHeads * 32, 0, st>>>(w.k, w.v, Ls, nch, w.part);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  coarse_kv_reduce_kernel<<<unsigned(n), kHeads * 32, 0, st>>>(w.part, nch, w.kv);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  coarse_attn_apply_kernel<<<dim3((Lx + kApplyTokens - 1) / kApplyTokens, unsigned(n)), kHeads * 32, 0, st>>>(
      w.q, w.kv, Lx, Ls, 1e-6f, w.msg);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  P = GemmParams{};
  P.mode[0] = EPI_LN; P.gamma = ln; P.beta = ln + kC;
  const Dst om[3] = {{w.m1, kC}, none, none};
  if ((e = gemm_run(Tx, w.msg, kC, nullptr, 0, wl + kOffMerge, 256, om, P, nullptr, st)) != cudaSuccess) return e;
  P = GemmParams{};
  P.mode[0] = EPI_RELU; P.mode[1] = EPI_RELU;
  const Dst oh[3] = {{w.hid, 2 * kC}, {w.hid + kC, 2 * kC}, none};
  if ((e = gemm_run(Tx, x, kC, w.m1, kC, wl + kOffMlp1, 512, oh, P, nullptr, st)) != cudaSuccess) return e;
  P = GemmParams{};
  P.mode[0] = EPI_LN_RES; P.gamma = ln + 2 * kC; P.beta = ln + 3 * kC;
  const Dst ox[3] = {{x, kC}, none, none};
  return gemm_run(Tx, w.hid, 2 * kC, nullptr, 0, wl + kOffMlp2, 256, ox, P, x, st);
}

// int32 row indices of the GEMM, and the attention grids' y dimension (one block row per pair)
bool too_many_rows(int64_t n, int L, int S) { return n > 65535 || n > (int64_t(0x7fffffff) - 2 * kTile) / (L > S ? L : S); }

}  // namespace
}  // namespace pope

using namespace pope;

extern "C" size_t pope_coarse_tf_workspace_bytes(int64_t n_pairs, int L, int S) {
  if (n_pairs <= 0 || L <= 0 || S <= 0 || too_many_rows(n_pairs, L, S)) return 0;
  return carve_coarse_tf(nullptr, n_pairs, L, S).bytes;
}

extern "C" int pope_coarse_transformer(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights,
                                       int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  if (!feat0 || !feat1 || !weights || !layer_kinds || !workspace) return POPE_ERR_INVALID_ARG;
  if (n_pairs < 0 || L <= 0 || S <= 0 || n_layers < 0) return POPE_ERR_INVALID_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (layer_kinds[l] != 0 && layer_kinds[l] != 1) return POPE_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(feat0) | reinterpret_cast<uintptr_t>(feat1) | reinterpret_cast<uintptr_t>(weights) |
       reinterpret_cast<uintptr_t>(workspace)) & 15u)
    return POPE_ERR_ALIGNMENT;
  if (too_many_rows(n_pairs, L, S)) return POPE_ERR_SHAPE;
  if (n_pairs == 0) return POPE_OK;
  const CoarseTfScratch w = carve_coarse_tf(workspace, n_pairs, L, S);
  if (workspace_bytes < w.bytes) return POPE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* x0 = static_cast<__nv_bfloat16*>(feat0);
  __nv_bfloat16* x1 = static_cast<__nv_bfloat16*>(feat1);
  for (int l = 0; l < n_layers; ++l) {
    const char* wl = static_cast<const char*>(weights) + size_t(l) * kLayerBytes;
    cudaError_t e;
    if (layer_kinds[l] == 0) {            // 'self'  (transformer.py:96-98)
      if ((e = encoder_layer(x0, x0, n_pairs, L, L, wl, w, st)) != cudaSuccess) return int(e);
      if ((e = encoder_layer(x1, x1, n_pairs, S, S, wl, w, st)) != cudaSuccess) return int(e);
    } else {                              // 'cross' (:99-101): feat1 attends to the UPDATED feat0
      if ((e = encoder_layer(x0, x1, n_pairs, L, S, wl, w, st)) != cudaSuccess) return int(e);
      if ((e = encoder_layer(x1, x0, n_pairs, S, L, wl, w, st)) != cudaSuccess) return int(e);
    }
  }
  return POPE_OK;
}

extern "C" int pope_coarse_pos_encode(const void* feat, const void* pe, int64_t n, int C, int H, int W, int pe_h, int pe_w,
                                      void* out, void* stream) {
  if (!feat || !pe || !out) return POPE_ERR_INVALID_ARG;
  if (n < 0 || H <= 0 || W <= 0 || pe_h <= 0 || pe_w <= 0) return POPE_ERR_INVALID_ARG;
  if (C != kC || H > pe_h || W > pe_w) return POPE_ERR_SHAPE;
  if (((reinterpret_cast<uintptr_t>(feat) | reinterpret_cast<uintptr_t>(pe)) & 3u) || (reinterpret_cast<uintptr_t>(out) & 15u))
    return POPE_ERR_ALIGNMENT;
  if (int64_t(H) * W > 0x7fffffff - kPePix || n > 65535) return POPE_ERR_SHAPE;
  if (n == 0) return POPE_OK;
  const int hw = H * W;
  coarse_pos_encode_kernel<<<dim3((hw + kPePix - 1) / kPePix, unsigned(n)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(feat), static_cast<const float*>(pe), H, W, pe_h, pe_w, static_cast<__nv_bfloat16*>(out));
  return int(cudaGetLastError());
}
