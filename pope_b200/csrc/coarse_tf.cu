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
//
// The same layer also runs at fp32 accuracy on the bf16 tensor cores (pope_coarse_transformer_f32): activations are fp32
// in HBM, every GEMM operand is split into three bf16 planes a = a1 + a2 + a3 (weights once when packed, activations by
// split3_kernel ahead of each GEMM), and coarse_gemm_kernel<true> accumulates the six significant products
// a1w1 + a2w1 + a3w1 + a1w2 + a2w2 + a1w3 of every k-chunk into the same fp32 TMEM accumulator (DESIGN §4.10).
#include <cuda.h>

#include <type_traits>

#include "common.cuh"
#include "split3.cuh"
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
// split (fp32-accuracy) form: an item's 256 output columns are computed as two N = 128 halves into the two halves of its
// accumulator, so that a stage holds the three A planes of a k-chunk and the three W planes of one half, six 16 KB boxes
// (three planes of a full 256-row W box next to three A boxes would be 144 KB a stage: no double buffering).  The A boxes
// are fetched once per half.  Two stages; epilogue staging is unchanged (a warp's fp32 box is 32 rows x 32 columns).
constexpr int kSplitStageBytes = 6 * kABytes;
constexpr int kSplitStages = 2;
constexpr int kSplitSmemAlloc = kSmemRing + kSplitStages * kSplitStageBytes + 1024;
static_assert(kSplitSmemAlloc <= 227 * 1024, "split coarse GEMM shared memory");
static_assert(kSmemTmemPtr + 16 <= kSmemRing && kSplitStages <= kStages, "the barrier block is sized for the bf16 ring");

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

// kSplit = false: bf16 activations and weights (2D maps), bf16 output rows.
// kSplit = true:  mapA0 / mapA1 / mapW are 3D maps over three bf16 planes (coordinate 2 = plane), output and residual rows
//                 are fp32 (32-column boxes).
template <bool kSplit>
__global__ void __launch_bounds__(kThreads, 1)
coarse_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                   const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapO0,
                   const __grid_constant__ CUtensorMap mapO1, const __grid_constant__ CUtensorMap mapO2,
                   const __grid_constant__ CUtensorMap mapR, const GemmParams P) {
  constexpr int kRing = kSplit ? kSplitStages : kStages;
  constexpr int kStage = kSplit ? kSplitStageBytes : kStageBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_full = sbase + kSmemBar, bar_empty = bar_full + 8 * kRing;
  const uint32_t bar_acc_full = bar_empty + 8 * kRing, bar_acc_empty = bar_acc_full + 16;
  const uint32_t bar_res = bar_acc_empty + 16;   // one per epilogue warp
  const uint32_t ring = sbase + kSmemRing;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kSmemTmemPtr);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (P.T + kTile - 1) / kTile, nitems = ntiles * P.ntn;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA0); prefetch_tmap(&mapA1); prefetch_tmap(&mapW);
    prefetch_tmap(&mapO0); prefetch_tmap(&mapO1); prefetch_tmap(&mapO2); prefetch_tmap(&mapR);
    for (int s = 0; s < kRing; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
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
          if constexpr (kSplit) {
            // stage = A planes 1-3 of the k-chunk, then W planes 1-3 of one 128-column half
            const CUtensorMap* ma = kc < P.ksplit ? &mapA0 : &mapA1;
            const int ka = (kc < P.ksplit ? kc : kc - P.ksplit) * kBoxK;
            for (int h = 0; h < 2; ++h) {
              mbar_wait(bar_empty + 8 * stage, phase ^ 1);
              const uint32_t dst = ring + stage * kStage;
              mbar_expect_tx(bar_full + 8 * stage, kStage);
              for (int p = 0; p < 3; ++p) tma_load_3d(dst + p * kABytes, ma, bar_full + 8 * stage, ka, t * kTile, p);
              for (int p = 0; p < 3; ++p)
                tma_load_3d(dst + (3 + p) * kABytes, &mapW, bar_full + 8 * stage, kc * kBoxK, j * kNTile + h * (kNTile / 2), p);
              if (++stage == kRing) { stage = 0; phase ^= 1; }
            }
          } else {
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            const uint32_t dst = ring + stage * kStage;
            mbar_expect_tx(bar_full + 8 * stage, kStage);
            if (kc < P.ksplit) tma_load_2d(dst, &mapA0, bar_full + 8 * stage, kc * kBoxK, t * kTile);
            else tma_load_2d(dst, &mapA1, bar_full + 8 * stage, (kc - P.ksplit) * kBoxK, t * kTile);
            tma_load_2d(dst + kABytes, &mapW, bar_full + 8 * stage, kc * kBoxK, j * kNTile);
            if (++stage == kRing) { stage = 0; phase ^= 1; }
          }
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
          if constexpr (kSplit) {
            constexpr uint32_t idesc_half = idesc_bf16(kTile, kNTile / 2);
            for (int h = 0; h < 2; ++h) {
              mbar_wait(bar_full + 8 * stage, phase);
              tc_fence_after();
              const uint32_t a_addr = ring + stage * kStage, b_addr = a_addr + 3 * kABytes;
              const uint32_t dh = d + h * (kNTile / 2);
              // a1w1 + a2w1 + a3w1 + a1w2 + a2w2 + a1w3 (plane of A, plane of W)
#pragma unroll
              for (int q = 0; q < 6; ++q) {
                const uint32_t pa = q == 1 || q == 4 ? 1u : (q == 2 ? 2u : 0u), pw = q < 3 ? 0u : (q < 5 ? 1u : 2u);
#pragma unroll
                for (int ks = 0; ks < kBoxK / 16; ++ks)
                  umma_bf16(dh, umma_desc(a_addr + pa * kABytes + ks * 32), umma_desc(b_addr + pw * kABytes + ks * 32),
                            idesc_half, (kc | q | ks) ? 1u : 0u);
              }
              umma_commit(bar_empty + 8 * stage);
              if (++stage == kRing) { stage = 0; phase ^= 1; }
            }
          } else {
            mbar_wait(bar_full + 8 * stage, phase);
            tc_fence_after();
            const uint32_t a_addr = ring + stage * kStage, b_addr = a_addr + kABytes;
#pragma unroll
            for (int ks = 0; ks < kBoxK / 16; ++ks)
              umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), idesc, (kc | ks) ? 1u : 0u);
            umma_commit(bar_empty + 8 * stage);                         // ring slot free once these MMAs have read it
            if (++stage == kRing) { stage = 0; phase ^= 1; }
          }
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
          if constexpr (kSplit) {        // fp32 accuracy: elu(x) + 1 as torch evaluates it (expm1, then + 1)
#pragma unroll
            for (int c = 0; c < 64; ++c) v[c] = v[c] > 0.f ? v[c] + 1.f : expm1f(v[c]) + 1.f;
          } else {
#pragma unroll
            for (int c = 0; c < 64; ++c) v[c] = v[c] > 0.f ? v[c] + 1.f : ex2_approx(v[c] * kLog2e);
          }
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
        if constexpr (kSplit) {          // fp32 rows: two boxes of 32 columns through the same 4 KB staging box
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            float* vh = v + hh * 32;
            if (lane == 0) tma_store_wait_read();
            __syncwarp();
            if (mode == EPI_LN_RES) {
              if (lane == 0) {
                mbar_expect_tx(bar_my_res, kStageOutBytes);
                tma_load_2d(stage_buf, &mapR, bar_my_res, col + hh * 32, row0);
              }
              __syncwarp();
              mbar_wait(bar_my_res, res_phase);
              res_phase ^= 1;
#pragma unroll
              for (int c8 = 0; c8 < 8; ++c8) {
                float4 r;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                             : "r"(my_row + ((uint32_t(c8) ^ sw) << 4)));
                vh[c8 * 4] += r.x; vh[c8 * 4 + 1] += r.y; vh[c8 * 4 + 2] += r.z; vh[c8 * 4 + 3] += r.w;
              }
              __syncwarp();
            }
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8)
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};"
                           ::"r"(my_row + ((uint32_t(c8) ^ sw) << 4)), "f"(vh[c8 * 4]), "f"(vh[c8 * 4 + 1]),
                             "f"(vh[c8 * 4 + 2]), "f"(vh[c8 * 4 + 3]) : "memory");
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(mo, stage_buf, col + hh * 32, row0);
              tma_store_commit();
            }
          }
          continue;
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

__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float to_f32(float x) { return x; }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }

// part[((b * nch + c) * kHeads + h) * kKvRows + e) * 32 + d]: e < 32 -> KV[d][e] over the chunk, e == 32 -> sum k[d]
// T: the activation type, __nv_bfloat16 or float
template <typename T>
__global__ void __launch_bounds__(kHeads * 32)
coarse_kv_partial_kernel(const T* __restrict__ k, const T* __restrict__ v, int S, int nch, float* __restrict__ part) {
  const int c = blockIdx.x, b = blockIdx.y, h = threadIdx.x >> 5, d = threadIdx.x & 31;
  const int s0 = c * kKvChunk, s1 = min(S, s0 + kKvChunk);
  float acc[kHeadDim], ks = 0.f;
#pragma unroll
  for (int e = 0; e < kHeadDim; ++e) acc[e] = 0.f;
  const T* kp = k + (size_t(b) * S + s0) * kC + h * kHeadDim + d;
  constexpr int kVec = kHeadDim * int(sizeof(T)) / 16;             // 16-byte vectors of one head's values
  const uint4* vp = reinterpret_cast<const uint4*>(v + (size_t(b) * S + s0) * kC + h * kHeadDim);
#pragma unroll 4
  for (int s = s0; s < s1; ++s, kp += kC, vp += kC * int(sizeof(T)) / 16) {
    const float kd = to_f32(*kp);
    uint4 q4[kVec];
#pragma unroll
    for (int i = 0; i < kVec; ++i) q4[i] = __ldg(vp + i);          // the same bytes in every lane: one broadcast
    if constexpr (std::is_same<T, float>::value) {
#pragma unroll
      for (int i = 0; i < kVec; ++i) {
        acc[4 * i] = fmaf(kd, __uint_as_float(q4[i].x), acc[4 * i]);
        acc[4 * i + 1] = fmaf(kd, __uint_as_float(q4[i].y), acc[4 * i + 1]);
        acc[4 * i + 2] = fmaf(kd, __uint_as_float(q4[i].z), acc[4 * i + 2]);
        acc[4 * i + 3] = fmaf(kd, __uint_as_float(q4[i].w), acc[4 * i + 3]);
      }
    } else {
      const uint32_t w[16] = {q4[0].x, q4[0].y, q4[0].z, q4[0].w, q4[1].x, q4[1].y, q4[1].z, q4[1].w,
                              q4[2].x, q4[2].y, q4[2].z, q4[2].w, q4[3].x, q4[3].y, q4[3].z, q4[3].w};
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        acc[2 * i] = fmaf(kd, bf_lo(w[i]), acc[2 * i]);
        acc[2 * i + 1] = fmaf(kd, bf_hi(w[i]), acc[2 * i + 1]);
      }
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
template <typename T>
__global__ void __launch_bounds__(kHeads * 32)
coarse_attn_apply_kernel(const T* __restrict__ q, const float* __restrict__ kv, int L, int S, float eps, T* __restrict__ msg) {
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
    const float ql = to_f32(q[off]);
    float o = 0.f, z = 0.f;
#pragma unroll
    for (int d = 0; d < kHeadDim; ++d) {
      const float qd = __shfl_sync(kFullMask, ql, d);
      o = fmaf(qd, kvc[d], o);
      z = fmaf(qd, ksum[d], z);
    }
    msg[off] = from_f32<T>(o * fs / (z + eps));
  }
}

// ---- position encoding + layout: out[b, y W + x, c] = T(feat[b, c, y, x] + pe[c, y, x]) ------------------------------
// T = __nv_bfloat16 (one round to nearest even) or float (the fp32 sum itself)
constexpr int kPePix = 32;

template <typename T>
__global__ void __launch_bounds__(256)
coarse_pos_encode_kernel(const float* __restrict__ feat, const float* __restrict__ pe, int H, int W, int pe_h, int pe_w,
                         T* __restrict__ out) {
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
  for (int pp = warp; pp < kPePix && p0 + pp < HW; pp += 8) {   // write one token row per warp
    T* o = out + (size_t(b) * HW + p0 + pp) * kC;
    if constexpr (sizeof(T) == 2) {                  // lane = 8 channels
      const float* r = &tile[pp][lane * 8];
      *reinterpret_cast<uint4*>(o + lane * 8) =
          make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
    } else {                                         // lane = 4 channels in each half of the row
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float* r = &tile[pp][h * (kC / 2) + lane * 4];
        *reinterpret_cast<float4*>(o + h * (kC / 2) + lane * 4) = make_float4(r[0], r[1], r[2], r[3]);
      }
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct Dst { void* ptr; int64_t pitch; };         // one 256-column output block (row pitch in elements)

template <bool kSplit>
cudaError_t gemm_launch(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mw, const CUtensorMap (&mo)[3],
                        const CUtensorMap& mr, int64_t T, int N, int K0, int K1, GemmParams P, cudaStream_t st) {
  constexpr int smem = kSplit ? kSplitSmemAlloc : kSmemAlloc;
  P.T = int(T);
  P.kchunks = (K0 + K1) / kBoxK;
  P.ksplit = K0 / kBoxK;
  P.ntn = N / kNTile;
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(coarse_gemm_kernel<kSplit>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess)
    return e;
  const int64_t nitems = (T + kTile - 1) / kTile * P.ntn;
  coarse_gemm_kernel<kSplit><<<unsigned(nitems < sms ? nitems : sms), kThreads, smem, st>>>(ma0, ma1, mw, mo[0], mo[1], mo[2],
                                                                                             mr, P);
  return cudaGetLastError();
}

bool bad_gemm_shape(int64_t T, int N, int K0, int K1) {
  return T > 0x7fffffff - kTile || N % kNTile || N / kNTile > 3 || K0 % kBoxK || K1 % kBoxK;
}

// Y[T, N] = epilogue(cat(A0[T, K0], A1[T, K1]) . W[N, K0 + K1]^T); out[j] receives output columns [256 j, 256 j + 256).
// resid (EPI_LN_RES): [T, 256] rows added after the LayerNorm.  bf16 activations, weights and output.
cudaError_t gemm_run(int64_t T, const void* A0, int K0, const void* A1, int K1, const void* W, int N, const Dst (&out)[3],
                     GemmParams P, const void* resid, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  const int K = K0 + K1;
  if (bad_gemm_shape(T, N, K0, K1)) return cudaErrorInvalidValue;
  CUtensorMap ma0, ma1, mw, mo[3], mr;
  if (!make_map2d(&ma0, A0, T, K0, K0)) return cudaErrorInvalidValue;
  if (!make_map2d(&ma1, K1 ? A1 : A0, T, K1 ? K1 : K0, K1 ? K1 : K0)) return cudaErrorInvalidValue;
  if (!make_map2d(&mw, W, N, K, K, kNTile)) return cudaErrorInvalidValue;
  for (int j = 0; j < 3; ++j) {
    const Dst& o = out[j < N / kNTile ? j : 0];   // unused maps still have to be valid descriptors
    if (!o.ptr || !make_map2d(&mo[j], o.ptr, T, kNTile, o.pitch, 32)) return cudaErrorInvalidValue;
  }
  if (!make_map2d(&mr, resid ? resid : out[0].ptr, T, kC, resid ? kC : out[0].pitch, 32)) return cudaErrorInvalidValue;
  return gemm_launch<false>(ma0, ma1, mw, mo, mr, T, N, K0, K1, P, st);
}

// the same at fp32 accuracy: A0, A1 and W as three bf16 planes each (split3), fp32 output and residual rows
cudaError_t gemm_run_split(int64_t T, Planes A0, int K0, Planes A1, int K1, Planes W, int N, const Dst (&out)[3],
                           GemmParams P, const float* resid, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (bad_gemm_shape(T, N, K0, K1)) return cudaErrorInvalidValue;
  CUtensorMap ma0, ma1, mw, mo[3], mr;
  if (!make_map_planes(&ma0, A0, T, K0, kTile)) return cudaErrorInvalidValue;
  if (!make_map_planes(&ma1, K1 ? A1 : A0, T, K1 ? K1 : K0, kTile)) return cudaErrorInvalidValue;
  if (!make_map_planes(&mw, W, N, K0 + K1, kNTile / 2)) return cudaErrorInvalidValue;
  for (int j = 0; j < 3; ++j) {
    const Dst& o = out[j < N / kNTile ? j : 0];
    if (!o.ptr || !make_map2d_f32(&mo[j], o.ptr, T, kNTile, o.pitch)) return cudaErrorInvalidValue;
  }
  if (!make_map2d_f32(&mr, resid ? resid : out[0].ptr, T, kC, resid ? kC : out[0].pitch)) return cudaErrorInvalidValue;
  return gemm_launch<true>(ma0, ma1, mw, mo, mr, T, N, K0, K1, P, st);
}

// packed weights of one d_model-256 LoFTREncoderLayer (byte offsets; matrices bf16 row-major [out, in] like nn.Linear)
constexpr size_t kOffQkv = 0;                                  // [768, 256]  q_proj, k_proj, v_proj stacked
constexpr size_t kOffMerge = kOffQkv + 768 * 256 * 2;          // [256, 256]
constexpr size_t kOffMlp1 = kOffMerge + 256 * 256 * 2;         // [512, 512]
constexpr size_t kOffMlp2 = kOffMlp1 + 512 * 512 * 2;          // [256, 512]
constexpr size_t kOffLn = kOffMlp2 + 256 * 512 * 2;            // fp32: norm1.weight, norm1.bias, norm2.weight, norm2.bias
constexpr size_t kLayerBytes = kOffLn + 4 * 256 * 4;
static_assert(kLayerBytes == POPE_COARSE_TF_LAYER_BYTES, "include/pope_b200.h documents this layout");
// the fp32 layout: the same order with every matrix as three consecutive bf16 planes (w = w1 + w2 + w3), so a matrix
// starts at 3x its bf16 offset and its planes lie one bf16 matrix apart
constexpr size_t kF32LayerBytes = 3 * kOffLn + 4 * 256 * 4;
static_assert(kF32LayerBytes == POPE_COARSE_TF_F32_LAYER_BYTES, "include/pope_b200.h documents this layout");

// bf16: five [n * max(L, S), 256] planes (q, k, v, msg, m1; the MLP's hidden [T, 512] spans the q and k planes, which are
// dead by then), the per-chunk KV partials and the reduced KV of every pair.  fp32: the same five planes in fp32, plus the
// split planes of the GEMM operands: three bf16 planes of x (xs) and a region of six [n * max(L, S), 256] bf16 units that
// holds, interleaved, the three planes of msg / LN1's output (ms, even units) and of a 'cross' layer's source (ss, odd
// units), and later the three [T, 512] planes of the hidden (two units each, from ms).
template <typename T>
struct CoarseTfScratch {
  T *q, *k, *v, *msg, *m1, *hid;
  __nv_bfloat16 *xs, *ms, *ss;
  size_t unit2;          // bytes of one bf16 [n * max(L, S), 256] unit
  float *part, *kv;
  int nch;
  size_t bytes;
};
template <typename T>
CoarseTfScratch<T> carve_coarse_tf(void* base, int64_t n, int L, int S) {
  CoarseTfScratch<T> w{};
  char* p = static_cast<char*>(base);
  const int lmax = L > S ? L : S;
  const size_t unit = align_up(size_t(n) * lmax * kC * sizeof(T), 256);
  w.nch = (lmax + kKvChunk - 1) / kKvChunk;
  size_t off = 0;
  w.q = reinterpret_cast<T*>(p + off); off += unit;
  w.k = reinterpret_cast<T*>(p + off); off += unit;
  w.v = reinterpret_cast<T*>(p + off); off += unit;
  w.msg = reinterpret_cast<T*>(p + off); off += unit;
  w.m1 = reinterpret_cast<T*>(p + off); off += unit;
  w.hid = w.q;
  if (sizeof(T) == 4) {
    w.unit2 = align_up(size_t(n) * lmax * kC * 2, 256);
    w.xs = reinterpret_cast<__nv_bfloat16*>(p + off); off += 3 * w.unit2;
    w.ms = reinterpret_cast<__nv_bfloat16*>(p + off);
    w.ss = reinterpret_cast<__nv_bfloat16*>(p + off + w.unit2); off += 6 * w.unit2;
  }
  w.part = reinterpret_cast<float*>(p + off); off += align_up(size_t(n) * w.nch * kKvFloats * 4, 256);
  w.kv = reinterpret_cast<float*>(p + off); off += align_up(size_t(n) * kKvFloats * 4, 256);
  w.bytes = off;
  return w;
}

// the global linear attention of one layer application: msg from q [n, Lx], k / v [n, Ls]
template <typename T>
cudaError_t attention(const CoarseTfScratch<T>& w, int64_t n, int Lx, int Ls, cudaStream_t st) {
  cudaError_t e;
  const int nch = (Ls + kKvChunk - 1) / kKvChunk;
  coarse_kv_partial_kernel<T><<<dim3(nch, unsigned(n)), kHeads * 32, 0, st>>>(w.k, w.v, Ls, nch, w.part);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  coarse_kv_reduce_kernel<<<unsigned(n), kHeads * 32, 0, st>>>(w.part, nch, w.kv);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  coarse_attn_apply_kernel<T><<<dim3((Lx + kApplyTokens - 1) / kApplyTokens, unsigned(n)), kHeads * 32, 0, st>>>(
      w.q, w.kv, Lx, Ls, 1e-6f, w.msg);
  return cudaGetLastError();
}

// x <- x + norm2(mlp(cat(x, norm1(merge(attention(q(x), k(src), v(src)))))))      (transformer.py:34-58), in place on x
// x: [n, Lx, 256], src: [n, Ls, 256]
cudaError_t encoder_layer(__nv_bfloat16* x, const __nv_bfloat16* src, int64_t n, int Lx, int Ls, const char* wl,
                          const CoarseTfScratch<__nv_bfloat16>& w, cudaStream_t st) {
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
  if ((e = attention(w, n, Lx, Ls, st)) != cudaSuccess) return e;
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

// the same layer on fp32 activations at fp32 accuracy: every GEMM operand is split into three bf16 planes first
cudaError_t encoder_layer(float* x, const float* src, int64_t n, int Lx, int Ls, const char* wl,
                          const CoarseTfScratch<float>& w, cudaStream_t st) {
  const int64_t Tx = n * Lx, Ts = n * Ls;
  const float* ln = reinterpret_cast<const float*>(wl + 3 * kOffLn);
  const Dst none{nullptr, 0};
  const Planes xs{w.xs, w.unit2}, ms{w.ms, 2 * w.unit2}, no{nullptr, 0};
  auto weight = [wl](size_t off, size_t rows, size_t cols) { return Planes{wl + 3 * off, rows * cols * 2}; };
  cudaError_t e;
  if ((e = split_planes(x, w.xs, xs.stride, size_t(Tx) * kC, st)) != cudaSuccess) return e;
  GemmParams P{};
  if (x == src) {
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_ELU1; P.mode[2] = EPI_SCALE; P.scale = 1.f / float(Ls);
    const Dst o[3] = {{w.q, kC}, {w.k, kC}, {w.v, kC}};
    if ((e = gemm_run_split(Tx, xs, kC, no, 0, weight(kOffQkv, 768, 256), 768, o, P, nullptr, st)) != cudaSuccess) return e;
  } else {
    const Planes ss{w.ss, 2 * w.unit2};
    if ((e = split_planes(src, w.ss, ss.stride, size_t(Ts) * kC, st)) != cudaSuccess) return e;
    P.mode[0] = EPI_ELU1;
    const Dst oq[3] = {{w.q, kC}, none, none};
    if ((e = gemm_run_split(Tx, xs, kC, no, 0, weight(kOffQkv, 768, 256), 256, oq, P, nullptr, st)) != cudaSuccess) return e;
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_SCALE; P.scale = 1.f / float(Ls);
    const Dst okv[3] = {{w.k, kC}, {w.v, kC}, none};
    Planes wkv = weight(kOffQkv, 768, 256);
    wkv.ptr = static_cast<const char*>(wkv.ptr) + 256 * 256 * 2;   // k_proj and v_proj rows of every plane
    if ((e = gemm_run_split(Ts, ss, kC, no, 0, wkv, 512, okv, P, nullptr, st)) != cudaSuccess) return e;
  }
  if ((e = attention(w, n, Lx, Ls, st)) != cudaSuccess) return e;
  if ((e = split_planes(w.msg, w.ms, ms.stride, size_t(Tx) * kC, st)) != cudaSuccess) return e;
  P = GemmParams{};
  P.mode[0] = EPI_LN; P.gamma = ln; P.beta = ln + kC;
  const Dst om[3] = {{w.m1, kC}, none, none};
  if ((e = gemm_run_split(Tx, ms, kC, no, 0, weight(kOffMerge, 256, 256), 256, om, P, nullptr, st)) != cudaSuccess) return e;
  if ((e = split_planes(w.m1, w.ms, ms.stride, size_t(Tx) * kC, st)) != cudaSuccess) return e;
  P = GemmParams{};
  P.mode[0] = EPI_RELU; P.mode[1] = EPI_RELU;
  const Dst oh[3] = {{w.hid, 2 * kC}, {w.hid + kC, 2 * kC}, none};
  if ((e = gemm_run_split(Tx, xs, kC, ms, kC, weight(kOffMlp1, 512, 512), 512, oh, P, nullptr, st)) != cudaSuccess) return e;
  if ((e = split_planes(w.hid, w.ms, ms.stride, size_t(Tx) * 2 * kC, st)) != cudaSuccess) return e;   // [T, 512] planes
  P = GemmParams{};
  P.mode[0] = EPI_LN_RES; P.gamma = ln + 2 * kC; P.beta = ln + 3 * kC;
  const Dst ox[3] = {{x, kC}, none, none};
  return gemm_run_split(Tx, ms, 2 * kC, no, 0, weight(kOffMlp2, 256, 512), 256, ox, P, x, st);
}

// int32 row indices of the GEMM, and the attention grids' y dimension (one block row per pair)
bool too_many_rows(int64_t n, int L, int S) { return n > 65535 || n > (int64_t(0x7fffffff) - 2 * kTile) / (L > S ? L : S); }

// T = __nv_bfloat16: pope_coarse_transformer; T = float: pope_coarse_transformer_f32
template <typename T>
int coarse_transformer(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights, int n_layers,
                       const int* layer_kinds, void* workspace, size_t workspace_bytes, void* stream) {
  constexpr size_t layer_bytes = sizeof(T) == 4 ? kF32LayerBytes : kLayerBytes;
  if (!feat0 || !feat1 || !weights || !layer_kinds || !workspace) return POPE_ERR_INVALID_ARG;
  if (n_pairs < 0 || L <= 0 || S <= 0 || n_layers < 0) return POPE_ERR_INVALID_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (layer_kinds[l] != 0 && layer_kinds[l] != 1) return POPE_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(feat0) | reinterpret_cast<uintptr_t>(feat1) | reinterpret_cast<uintptr_t>(weights) |
       reinterpret_cast<uintptr_t>(workspace)) & 15u)
    return POPE_ERR_ALIGNMENT;
  if (too_many_rows(n_pairs, L, S)) return POPE_ERR_SHAPE;
  if (n_pairs == 0) return POPE_OK;
  const CoarseTfScratch<T> w = carve_coarse_tf<T>(workspace, n_pairs, L, S);
  if (workspace_bytes < w.bytes) return POPE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  T* x0 = static_cast<T*>(feat0);
  T* x1 = static_cast<T*>(feat1);
  for (int l = 0; l < n_layers; ++l) {
    const char* wl = static_cast<const char*>(weights) + size_t(l) * layer_bytes;
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

}  // namespace
}  // namespace pope

using namespace pope;

extern "C" size_t pope_coarse_tf_workspace_bytes(int64_t n_pairs, int L, int S) {
  if (n_pairs <= 0 || L <= 0 || S <= 0 || too_many_rows(n_pairs, L, S)) return 0;
  return carve_coarse_tf<__nv_bfloat16>(nullptr, n_pairs, L, S).bytes;
}

extern "C" size_t pope_coarse_tf_f32_workspace_bytes(int64_t n_pairs, int L, int S) {
  if (n_pairs <= 0 || L <= 0 || S <= 0 || too_many_rows(n_pairs, L, S)) return 0;
  return carve_coarse_tf<float>(nullptr, n_pairs, L, S).bytes;
}

extern "C" int pope_coarse_transformer(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights,
                                       int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  return coarse_transformer<__nv_bfloat16>(feat0, feat1, n_pairs, L, S, weights, n_layers, layer_kinds, workspace,
                                           workspace_bytes, stream);
}

extern "C" int pope_coarse_transformer_f32(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights,
                                           int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  return coarse_transformer<float>(feat0, feat1, n_pairs, L, S, weights, n_layers, layer_kinds, workspace, workspace_bytes,
                                   stream);
}

extern "C" int pope_coarse_pos_encode_ex(const void* feat, const void* pe, int64_t n, int C, int H, int W, int pe_h,
                                         int pe_w, void* out, int out_dtype, void* stream) {
  if (!feat || !pe || !out) return POPE_ERR_INVALID_ARG;
  if (n < 0 || H <= 0 || W <= 0 || pe_h <= 0 || pe_w <= 0) return POPE_ERR_INVALID_ARG;
  if (out_dtype != POPE_BF16 && out_dtype != POPE_F32) return POPE_ERR_DTYPE;
  if (C != kC || H > pe_h || W > pe_w) return POPE_ERR_SHAPE;
  if (((reinterpret_cast<uintptr_t>(feat) | reinterpret_cast<uintptr_t>(pe)) & 3u) || (reinterpret_cast<uintptr_t>(out) & 15u))
    return POPE_ERR_ALIGNMENT;
  if (int64_t(H) * W > 0x7fffffff - kPePix || n > 65535) return POPE_ERR_SHAPE;
  if (n == 0) return POPE_OK;
  const int hw = H * W;
  const dim3 grid((hw + kPePix - 1) / kPePix, unsigned(n));
  const float* f = static_cast<const float*>(feat);
  const float* p = static_cast<const float*>(pe);
  if (out_dtype == POPE_BF16)
    coarse_pos_encode_kernel<__nv_bfloat16><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        f, p, H, W, pe_h, pe_w, static_cast<__nv_bfloat16*>(out));
  else
    coarse_pos_encode_kernel<float><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(f, p, H, W, pe_h, pe_w,
                                                                                          static_cast<float*>(out));
  return int(cudaGetLastError());
}

extern "C" int pope_coarse_pos_encode(const void* feat, const void* pe, int64_t n, int C, int H, int W, int pe_h, int pe_w,
                                      void* out, void* stream) {
  return pope_coarse_pos_encode_ex(feat, pe, n, C, H, W, pe_h, pe_w, out, POPE_BF16, stream);
}
