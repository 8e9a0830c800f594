// fine_tf.cu -- the fine-level LoFTR transformer and the FinePreprocess Linears on sm_100a (SURVEY.md 8(f), rank 1).
//
// Replaces, for bf16 windows, the op sequence of the reference's
//   src/matcher/loftr_module/transformer.py:34-58      (LoFTREncoderLayer.forward: q/k/v projections, linear attention,
//                                                       merge, LayerNorm, 2-layer MLP on cat(x, message), LayerNorm, residual)
//   src/matcher/loftr_module/linear_attention.py:21-47 (elu(x)+1 feature map, KV = K^T V / S, Z = 1/(Q . sum K + eps))
//   src/matcher/loftr_module/transformer.py:95-104     ('self' / 'cross' layer schedule)
//   src/matcher/loftr_module/fine_preprocess.py:50-57  (down_proj of the matched coarse features, merge_feat on
//                                                       cat(window, coarse))
// Every Linear outside the encoder MLP is one launch of linear_tc_kernel: a persistent, weight-stationary tcgen05 GEMM
// (the whole weight matrix stays in shared memory, 128-token tiles of the activations stream through a TMA ring,
// accumulators in TMEM) whose epilogue applies what follows the Linear in the reference (feature map, 1/S scale,
// LayerNorm, bias, per-window vector) before the row is written back as bf16.  The encoder MLP (both Linears, the ReLU
// between them, LayerNorm2 and the residual) is one launch of mlp_fused_kernel.  The attention itself (8 heads x 16 x 16
// per window) is a warp-per-window kernel: mma.sync tensor cores for windows of at most 32 tokens, fp32 SIMT above.
// Activations are bf16 in HBM, all arithmetic accumulates in fp32.
#include <cuda.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace pope {
namespace {

using namespace tc1;

constexpr int kD = 128;                  // fine d_model
constexpr int kHeads = 8, kHeadDim = 16;
constexpr int kTile = 128;               // token rows per tile (MMA M)
constexpr int kBoxK = 64;                // bf16 elements per 128-byte swizzle row
constexpr int kBoxBytes = kTile * kBoxK * 2;          // 16384
constexpr int kMaxWBoxes = 8;            // N/128 * K/64 <= 8 (256 x 256)
constexpr int kMaxStages = 8;            // activation ring depth (as many as fit beside the weights)
constexpr int kSlots = 4;                // TMEM accumulator slots of 128 columns
constexpr int kEpiWarps = 8;             // two sets of four (one warp per TMEM lane quadrant); sets alternate items
constexpr int kLinThreads = 64 + kEpiWarps * 32;      // warp 0: TMA, warp 1: MMA, warps 2-9: epilogue
constexpr int kStageOutBytes = 32 * 128;              // per epilogue warp: 32 rows x 64 bf16 columns, 128B-swizzled
constexpr int kSmemBudget = 227 * 1024 - 1024;        // dynamic shared memory we ask for (1 KB alignment slack inside)
// layout: [staging: 8 x 4 KB][barriers][weights: nbox x 16 KB][ring: stages x 16 KB]
constexpr int kSmemOut = 0;
constexpr int kSmemBar = kSmemOut + kEpiWarps * kStageOutBytes;
constexpr int kNumBars = 1 + 2 * kMaxStages + 2 * kSlots;
constexpr int kSmemTmemPtr = kSmemBar + kNumBars * 8;
constexpr int kSmemW = 34 * 1024;                     // 1024-aligned, past the barriers (sets the ring depth below)
static_assert(kSmemTmemPtr + 16 <= kSmemW, "barrier block overlaps the weights");
constexpr int kSmemAlloc = kSmemBudget;               // > 113 KB -> one CTA per SM, so the CTA may take all 512 TMEM columns

enum EpiMode : int { EPI_COPY = 0, EPI_ELU1 = 1, EPI_SCALE = 2, EPI_LN = 3, EPI_ADDVEC = 4 };

struct LinParams {
  int T;                       // token rows
  int kchunks;                 // K/64
  int nblk;                    // N/128
  int stages;                  // ring depth that fits beside the weights
  float* out_f32;              // if set: the (single) output block is written as fp32 rows [T, 128] with plain stores
  int mode[3];
  float scale;                 // EPI_SCALE
  const float* bias;           // [N] or nullptr, added before the mode is applied
  const float* gamma;          // EPI_LN: [128]
  const float* beta;
  const float* rowvec;         // EPI_ADDVEC: [T / rows_per_vec, 128]
  int rows_per_vec;
  const int32_t* live;         // if set: device count of live items; rows >= *live * rows_per_item are not written and
  int rows_per_item;           // tiles past them not run (T is the capacity the tensor maps and the grid are sized for)
  __nv_bfloat16* out_rows[3];  // output blocks as plain pointers (row pitch out_pitch), for the one 32-row box that
  int out_pitch[3];            // straddles the live bound: a TMA store of it would write rows past the bound
};

// Live part of a capacity-sized launch: cap, or min(cap, *live * per_item) when a device count is given.  Every kernel
// reads the count once, at its start; it is written by an earlier kernel in stream order.  (None of these kernels uses
// programmatic dependent launch; one that does must read it after griddepcontrol.wait.)
__device__ __forceinline__ int64_t live_count(int64_t cap, const int32_t* live, int64_t per_item) {
  return live ? min(cap, int64_t(max(*live, 0)) * per_item) : cap;
}

// A 32-row output box that straddles the live bound is not TMA-stored (the store would write the rows past the bound):
// each lane below the bound copies its own 64-column half row out of the 128B-swizzled staging box instead.
__device__ __forceinline__ void store_staged_half_row(uint32_t my_row, uint32_t sw, __nv_bfloat16* dst) {
#pragma unroll
  for (int c8 = 0; c8 < 8; ++c8) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "r"(my_row + ((uint32_t(c8) ^ sw) << 4)));
    reinterpret_cast<uint4*>(dst)[c8] = r;
  }
}

// mapX: activations [T, K]; mapO[j]: output block j as a [T, 128] bf16 tensor (box 64 x 32 rows).
// kBounded: P.live is set (a separate instantiation, so that the unbounded launches keep their code and registers)
template <bool kBounded>
__global__ void __launch_bounds__(kLinThreads, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
                 const __grid_constant__ CUtensorMap mapO0, const __grid_constant__ CUtensorMap mapO1,
                 const __grid_constant__ CUtensorMap mapO2, const LinParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + kSmemBar;
  const uint32_t bar_w_full = bar0;
  const uint32_t bar_x_full = bar0 + 8, bar_x_empty = bar_x_full + 8 * kMaxStages;
  const uint32_t bar_acc_full = bar_x_empty + 8 * kMaxStages, bar_acc_empty = bar_acc_full + 8 * kSlots;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kSmemTmemPtr);
  // live rows: read into shared memory once, so the epilogue re-reads it where needed instead of holding a register
  volatile int* live_rows_smem = reinterpret_cast<volatile int*>(smem + kSmemTmemPtr + 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int ntiles;
  {
    const int T = kBounded ? int(live_count(P.T, P.live, P.rows_per_item)) : P.T;
    ntiles = (T + kTile - 1) / kTile;
    if (kBounded) {
      if (int(blockIdx.x) >= ntiles) return;         // capacity-sized grid, fewer live tiles: no load issued, no TMEM held
      if (threadIdx.x == 0) *live_rows_smem = T;     // (every thread read the same count; published by the sync below)
    }
  }
  const uint32_t smem_x = sbase + kSmemW + P.nblk * P.kchunks * kBoxBytes;
  const int stages = P.stages;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapX); prefetch_tmap(&mapW);
    prefetch_tmap(&mapO0); prefetch_tmap(&mapO1); prefetch_tmap(&mapO2);
    mbar_init(bar_w_full, 1);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(bar_x_full + 8 * s, 1); mbar_init(bar_x_empty + 8 * s, 1); }
    for (int s = 0; s < kSlots; ++s) { mbar_init(bar_acc_full + 8 * s, 1); mbar_init(bar_acc_empty + 8 * s, 4); }
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
      mbar_expect_tx(bar_w_full, uint32_t(P.nblk * P.kchunks * kBoxBytes));
      for (int j = 0; j < P.nblk; ++j)
        for (int kc = 0; kc < P.kchunks; ++kc)
          tma_load_2d(sbase + kSmemW + (j * P.kchunks + kc) * kBoxBytes, &mapW, bar_w_full, kc * kBoxK, j * kTile);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x)
        for (int kc = 0; kc < P.kchunks; ++kc) {
          mbar_wait(bar_x_empty + 8 * stage, phase ^ 1);
          mbar_expect_tx(bar_x_full + 8 * stage, kBoxBytes);
          tma_load_2d(smem_x + stage * kBoxBytes, &mapX, bar_x_full + 8 * stage, kc * kBoxK, t * kTile);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16(kTile, 128);
      mbar_wait(bar_w_full, 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0, item = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        for (int j = 0; j < P.nblk; ++j) {                      // the tile's accumulator slots must have been drained
          const uint32_t it = item + j;
          mbar_wait(bar_acc_empty + 8 * (it & (kSlots - 1)), ((it / kSlots) & 1) ^ 1);
        }
        tc_fence_after();
        for (int kc = 0; kc < P.kchunks; ++kc) {
          mbar_wait(bar_x_full + 8 * stage, phase);
          tc_fence_after();
          const uint32_t a_addr = smem_x + stage * kBoxBytes;
          for (int j = 0; j < P.nblk; ++j) {
            const uint32_t d = tmem_base + ((item + j) & (kSlots - 1)) * 128;
            const uint32_t b_addr = sbase + kSmemW + (j * P.kchunks + kc) * kBoxBytes;
#pragma unroll
            for (int ks = 0; ks < kBoxK / 16; ++ks)
              umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), idesc, (kc | ks) ? 1u : 0u);
          }
          umma_commit(bar_x_empty + 8 * stage);                 // ring slot free once these MMAs have read it
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        for (int j = 0; j < P.nblk; ++j) umma_commit(bar_acc_full + 8 * ((item + j) & (kSlots - 1)));
        item += P.nblk;
      }
    }
  } else {
    // =============================== epilogue: thread = token row, 128 channels in registers =========================
    // Rows leave through a 128B-swizzled shared-memory box and a TMA store (a thread-per-row store to global memory
    // touches 32 different lines per instruction and was measured LSU-bound).
    const int ew = warp - 2, set = ew >> 2, quad = warp & 3;
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    const uint32_t stage_buf = sbase + kSmemOut + ew * kStageOutBytes;
    const uint32_t my_row = stage_buf + lane * 128;
    const uint32_t sw = uint32_t(lane & 7);
    // my_row is 128-byte aligned, so chunk c8 of the row sits at my_row_sw ^ (c8 << 4): one LOP3 per store, which keeps
    // ptxas from holding the eight chunk addresses across the item loop (at the 168-register cap it spilled them)
    const uint32_t my_row_sw = my_row + (sw << 4);
    uint32_t item = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int row0 = t * kTile + quad * 32, row = row0 + lane;
      for (int j = 0; j < P.nblk; ++j, ++item) {
        if ((item & 1u) != uint32_t(set)) continue;
        const uint32_t slot = item & (kSlots - 1);
        const int mode = P.mode[j];
        mbar_wait(bar_acc_full + 8 * slot, (item / kSlots) & 1);
        tc_fence_after();
        float v[kD];
        tmem_ld128(tmem_base + lane_addr + slot * 128, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty + 8 * slot);
        if (P.bias) {
          const float4* b4 = reinterpret_cast<const float4*>(P.bias + j * kD);
#pragma unroll
          for (int c = 0; c < kD; c += 4) {
            const float4 b = __ldg(b4 + (c >> 2));
            v[c] += b.x; v[c + 1] += b.y; v[c + 2] += b.z; v[c + 3] += b.w;
          }
        }
        if (mode == EPI_ELU1) {
#pragma unroll
          for (int c = 0; c < kD; ++c) v[c] = v[c] > 0.f ? v[c] + 1.f : ex2_approx(v[c] * kLog2e);
        } else if (mode == EPI_SCALE) {
#pragma unroll
          for (int c = 0; c < kD; ++c) v[c] *= P.scale;
        } else if (mode == EPI_LN) {
          float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
          for (int c = 0; c < kD; c += 4) { s0 += v[c]; s1 += v[c + 1]; s2 += v[c + 2]; s3 += v[c + 3]; }
          const float mean = ((s0 + s1) + (s2 + s3)) * (1.f / kD);
          s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
          for (int c = 0; c < kD; c += 4) {
            const float d0 = v[c] - mean, d1 = v[c + 1] - mean, d2 = v[c + 2] - mean, d3 = v[c + 3] - mean;
            s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
          }
          const float rstd = rsqrtf(((s0 + s1) + (s2 + s3)) * (1.f / kD) + 1e-5f);      // nn.LayerNorm: biased variance
          const float4* g4 = reinterpret_cast<const float4*>(P.gamma);
          const float4* b4 = reinterpret_cast<const float4*>(P.beta);
#pragma unroll
          for (int c = 0; c < kD; c += 4) {
            const float4 g = __ldg(g4 + (c >> 2)), b = __ldg(b4 + (c >> 2));
            v[c] = fmaf((v[c] - mean) * rstd, g.x, b.x); v[c + 1] = fmaf((v[c + 1] - mean) * rstd, g.y, b.y);
            v[c + 2] = fmaf((v[c + 2] - mean) * rstd, g.z, b.z); v[c + 3] = fmaf((v[c + 3] - mean) * rstd, g.w, b.w);
          }
        } else if (mode == EPI_ADDVEC) {
          if (row < (kBounded ? *live_rows_smem : P.T)) {
            const float4* a4 = reinterpret_cast<const float4*>(P.rowvec + size_t(row / P.rows_per_vec) * kD);
#pragma unroll
            for (int c = 0; c < kD; c += 4) {
              const float4 a = __ldg(a4 + (c >> 2));
              v[c] += a.x; v[c + 1] += a.y; v[c + 2] += a.z; v[c + 3] += a.w;
            }
          }
        }
        if (P.out_f32) {
          if (row < (kBounded ? *live_rows_smem : P.T)) {
            float4* o = reinterpret_cast<float4*>(P.out_f32 + size_t(row) * kD);
#pragma unroll
            for (int c = 0; c < kD; c += 4) o[c >> 2] = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
          }
        } else {
          const CUtensorMap* mo = j == 0 ? &mapO0 : (j == 1 ? &mapO1 : &mapO2);
          const int T = kBounded ? *live_rows_smem : P.T;
          const bool whole_box = !kBounded || row0 + 32 <= T || T == P.T;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            if (lane == 0) tma_store_wait_read();               // the previous store out of this box has read it
            __syncwarp();
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8) {
              const int c = half * 64 + c8 * 8;
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                           ::"r"(my_row_sw ^ (uint32_t(c8) << 4)), "r"(pack_bf16(v[c], v[c + 1])),
                             "r"(pack_bf16(v[c + 2], v[c + 3])), "r"(pack_bf16(v[c + 4], v[c + 5])),
                             "r"(pack_bf16(v[c + 6], v[c + 7])) : "memory");
            }
            fence_proxy_async();
            __syncwarp();
            if (whole_box) {
              if (lane == 0) {
                tma_store_2d(mo, stage_buf, half * 64, row0);   // rows past the capacity are clipped by the tensor map
                tma_store_commit();
              }
            } else {
              if (row < T) store_staged_half_row(my_row, sw, P.out_rows[j] + size_t(row) * P.out_pitch[j] + half * 64);
              __syncwarp();                                     // every lane has read its row before the box is refilled
            }
          }
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

// ---- fused MLP: x <- x + LayerNorm2(W2 . relu(W1 . cat(x, m1)))   (transformer.py:52-58) ---------------------------------
// One CTA PAIR per 256 token rows (cta_group::2, 128 rows per CTA).  Both weight matrices stay resident, split across the
// pair along their output dimension (W1: 2 x 128 of 256 rows, W2: 2 x 64 of 128 rows), which is what makes them fit:
//   MMA 1   D1[256 x 256] = cat(x, m1) . W1^T     (x / m1 tiles stream through a TMA ring; K = 256)
//   epi 1   relu(D1) -> bf16 -> the hidden tile h, written straight into shared memory in the K-major 128B-swizzled
//           operand layout (never to HBM: saves 4 of the 8 activation planes two separate Linear launches would move)
//   MMA 2   D2[256 x 128] = h . W2^T
//   epi 2   LayerNorm2, + x (residual rows by TMA), bf16, TMA store in place
// warp 0: TMA producer, warp 1: TMEM allocator + MMA issuer (leader CTA), warps 2-5: epilogue 2 of every tile, warps 6-9:
// epilogue 1 of every tile (four lane quadrants each), so epilogue 2 of tile t overlaps epilogue 1 of tile t+1.
// TMEM holds two 256-column buffers: buffer (tile & 1) receives D1 of its tile and, once epilogue 1 has drained it, D2
// of the same tile, so MMA 1 of tile t+1 runs while tile t is in epilogue 1; h is single-buffered).
namespace fm {
constexpr int kFmThreads = 320;
constexpr int kFmStages = 3;
constexpr int kW2BoxBytes = 64 * kBoxK * 2;                     // 64 rows (N/2 per CTA) x 64 k = 8 KB
constexpr int kFmOut = 0;                                      // 4 x 4 KB staging boxes (epilogue-2 warps)
constexpr int kFmBar = 4 * kStageOutBytes;                     // 16 KB
constexpr int kFmW1 = 17 * 1024;                               // 4 k-chunks x 16 KB
constexpr int kFmW2 = kFmW1 + 4 * kBoxBytes;                 // 4 k-chunks x 8 KB
constexpr int kFmH = kFmW2 + 4 * kW2BoxBytes;                // 4 k-chunks x 16 KB
constexpr int kFmX = kFmH + 4 * kBoxBytes;                   // kFmStages x 16 KB
constexpr int kFmEnd = kFmX + kFmStages * kBoxBytes;
constexpr int kFmTmemPtr = kFmBar + 64 * 8;
static_assert(kFmTmemPtr + 16 <= kFmW1 && kFmEnd + 1024 <= 227 * 1024, "fused-MLP shared memory layout");
constexpr int kFmAlloc = kFmEnd + 1024;
}  // namespace fm

template <bool kBounded>                                         // as linear_tc_kernel
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(fm::kFmThreads, 1)
mlp_fused_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapM1,
                 const __grid_constant__ CUtensorMap mapW1, const __grid_constant__ CUtensorMap mapW2,
                 const __grid_constant__ CUtensorMap mapO, const __grid_constant__ CUtensorMap mapR, int T_cap,
                 const int32_t* live, int rows_per_item, __nv_bfloat16* __restrict__ out,
                 const float* __restrict__ gamma, const float* __restrict__ beta) {
  using namespace fm;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + kFmBar;
  const uint32_t bar_w_full = bar0;
  const uint32_t bar_x_full = bar0 + 8, bar_x_empty = bar_x_full + 8 * kFmStages;
  // d1_full / d2_full exist once per epilogue set (even / odd tiles): a parity wait must see every phase of its barrier
  const uint32_t bar_d1_full = bar_x_empty + 8 * kFmStages, bar_h_full = bar_d1_full + 16;
  const uint32_t bar_d2_full = bar_h_full + 8, bar_d2_empty = bar_d2_full + 16;      // d2_empty: one per TMEM buffer
  const uint32_t bar_res = bar_d2_empty + 16;                    // 8: one per epilogue warp
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kFmTmemPtr);
  volatile int* live_rows_smem = reinterpret_cast<volatile int*>(smem + kFmTmemPtr + 8);   // as in linear_tc_kernel
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = tc2::cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  int ntiles;                                                    // 256-row tiles
  {
    const int T = kBounded ? int(live_count(T_cap, live, rows_per_item)) : T_cap;
    ntiles = (T + 2 * kTile - 1) / (2 * kTile);
    if (kBounded) {
      if (pair >= ntiles) return;      // both CTAs of the pair read the same count: neither issues a load nor allocates
      if (threadIdx.x == 0) *live_rows_smem = T;
    }
  }

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapX); prefetch_tmap(&mapM1); prefetch_tmap(&mapW1); prefetch_tmap(&mapW2);
    prefetch_tmap(&mapO); prefetch_tmap(&mapR);
    mbar_init(bar_w_full, 1);
    for (int s = 0; s < kFmStages; ++s) { mbar_init(bar_x_full + 8 * s, 1); mbar_init(bar_x_empty + 8 * s, 1); }
    mbar_init(bar_d1_full, 1); mbar_init(bar_d1_full + 8, 1);
    mbar_init(bar_h_full, 8);                                    // the 4 epilogue-1 warps of each CTA; leader's copy is used
    mbar_init(bar_d2_full, 1); mbar_init(bar_d2_full + 8, 1);
    mbar_init(bar_d2_empty, 8); mbar_init(bar_d2_empty + 8, 8);  // likewise
    for (int s = 0; s < 8; ++s) mbar_init(bar_res + 8 * s, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tc2::tmem_alloc(sbase + kFmTmemPtr, 512u);
    tc2::tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc2::cluster_sync_all();                                       // peer barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // =============================== TMA producer (both CTAs) ===============================
    if (lane == 0) {
      if (rank == 0) mbar_expect_tx(bar_w_full, 2 * (4 * kBoxBytes + 4 * kW2BoxBytes));
      for (int kc = 0; kc < 4; ++kc) {
        tc2::tma_load_2d_2sm(sbase + kFmW1 + kc * kBoxBytes, &mapW1, bar_w_full, kc * kBoxK, int(rank) * 128);
        tc2::tma_load_2d_2sm(sbase + kFmW2 + kc * kW2BoxBytes, &mapW2, bar_w_full, kc * kBoxK, int(rank) * 64);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair; t < ntiles; t += npairs) {
        const int row0 = t * 2 * kTile + int(rank) * kTile;
        for (int kc = 0; kc < 4; ++kc) {
          mbar_wait(bar_x_empty + 8 * stage, phase ^ 1);
          if (rank == 0) mbar_expect_tx(bar_x_full + 8 * stage, 2 * kBoxBytes);
          tc2::tma_load_2d_2sm(sbase + kFmX + stage * kBoxBytes, kc < 2 ? &mapX : &mapM1, bar_x_full + 8 * stage,
                               (kc & 1) * kBoxK, row0);
          if (++stage == kFmStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (leader CTA) ===============================
    if (rank == 0 && lane == 0) {
      constexpr uint32_t idesc1 = tc2::idesc_bf16_m256(256), idesc2 = tc2::idesc_bf16_m256(128);
      mbar_wait(bar_w_full, 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t n_it = pair < ntiles ? uint32_t((ntiles - 1 - pair) / npairs + 1) : 0u;
      // Two instruction streams share the tensor pipe: MMA 1 of tile it1 (D1 -> TMEM buffer it1 & 1, free once epilogue 2
      // of tile it1 - 2 has read its D2; one 64-wide k-chunk per ring stage) and MMA 2 of tile it2 <= it1 (needs the
      // hidden tile).  The issuer polls: MMA 2 goes first whenever its operands are ready (it unblocks epilogue 2 and
      // the reuse of h), otherwise the next chunk of MMA 1 whose ring stage has landed, at most one tile ahead.
      uint32_t it1 = 0, it2 = 0;
      int kc1 = 0;
      const long long t0 = clock64();
      uint32_t spins = 0;
      while (it2 < n_it) {
        bool progressed = false;
        if (it2 < it1 && mbar_try_wait(bar_h_full, it2 & 1)) {
          tc_fence_after();
          const uint32_t d = tmem_base + (it2 & 1) * 256;
          for (int kc = 0; kc < 4; ++kc) {
            const uint32_t a_addr = sbase + kFmH + kc * kBoxBytes, b_addr = sbase + kFmW2 + kc * kW2BoxBytes;
#pragma unroll
            for (int ks = 0; ks < kBoxK / 16; ++ks)
              tc2::umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), idesc2, (kc | ks) ? 1u : 0u);
          }
          tc2::umma_commit(bar_d2_full + 8 * (it2 & 1));
          ++it2;
          progressed = true;
        }
        if (it1 < n_it && it1 <= it2 + 1 &&
            (kc1 > 0 || mbar_try_wait(bar_d2_empty + 8 * (it1 & 1), ((it1 >> 1) & 1) ^ 1)) &&
            mbar_try_wait(bar_x_full + 8 * stage, phase)) {
          tc_fence_after();
          const uint32_t d = tmem_base + (it1 & 1) * 256;
          const uint32_t a_addr = sbase + kFmX + stage * kBoxBytes, b_addr = sbase + kFmW1 + kc1 * kBoxBytes;
#pragma unroll
          for (int ks = 0; ks < kBoxK / 16; ++ks)
            tc2::umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), idesc1, (kc1 | ks) ? 1u : 0u);
          tc2::umma_commit(bar_x_empty + 8 * stage);
          if (++stage == kFmStages) { stage = 0; phase ^= 1; }
          if (++kc1 == 4) {
            tc2::umma_commit(bar_d1_full + 8 * (it1 & 1));
            kc1 = 0;
            ++it1;
          }
          progressed = true;
        }
        if (progressed) spins = 0;
        else if ((++spins & 1023u) == 0 && clock64() - t0 > 8000000000ll) __trap();     // never hang the GPU
      }
    }
  } else {
    // =============================== epilogue ===============================
    const int ew = warp - 2, set = ew >> 2, quad = warp & 3;
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    const int rin = quad * 32 + lane;                            // row of this CTA's 128-row tile
    const uint32_t sw = uint32_t(lane & 7);
    const uint32_t stage_buf = sbase + kFmOut + quad * kStageOutBytes;        // epilogue-2 warps only
    const uint32_t my_row = stage_buf + lane * 128;
    const uint32_t bar_my_res = bar_res + 8 * quad;
    uint32_t res_phase = 0, it = 0;
    for (int t = pair; t < ntiles; t += npairs, ++it) {
      const int row0 = t * 2 * kTile + int(rank) * kTile + quad * 32;
      if (set == 1) {
      // ---- epilogue 1 (warps 6-9): relu(D1) -> h (4 k-chunks of 64 hidden columns) -----------------------------------
      mbar_wait(bar_d1_full + 8 * (it & 1), (it >> 1) & 1);
      if (it > 0) mbar_wait(bar_d2_full + 8 * ((it - 1) & 1), ((it - 1) >> 1) & 1);   // MMA 2 of the previous tile no longer reads h
      tc_fence_after();
#pragma unroll 1
      for (int hb = 0; hb < 2; ++hb) {                           // 128 hidden columns per pass: one TMEM round trip
        float v[kD];
        tmem_ld128(tmem_base + (it & 1) * 256 + lane_addr + hb * 128, v);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const uint32_t hrow = sbase + kFmH + (2 * hb + half) * kBoxBytes + uint32_t(rin) * 128;
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) {
            const int c = half * 64 + c8 * 8;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                         ::"r"(hrow + ((uint32_t(c8) ^ sw) << 4)), "r"(pack_bf16(fmaxf(v[c], 0.f), fmaxf(v[c + 1], 0.f))),
                           "r"(pack_bf16(fmaxf(v[c + 2], 0.f), fmaxf(v[c + 3], 0.f))),
                           "r"(pack_bf16(fmaxf(v[c + 4], 0.f), fmaxf(v[c + 5], 0.f))),
                           "r"(pack_bf16(fmaxf(v[c + 6], 0.f), fmaxf(v[c + 7], 0.f))) : "memory");
          }
        }
      }
      fence_proxy_async();                                       // the MMA reads h through the async proxy
      tc_fence_before();
      __syncwarp();
      if (lane == 0) tc2::mbar_arrive_leader_release(bar_h_full);
      continue;
      }
      // ---- epilogue 2 (warps 2-5): LayerNorm2(D2) + x -> out ------------------------------------------------------------
      mbar_wait(bar_d2_full + 8 * (it & 1), (it >> 1) & 1);
      tc_fence_after();
      float v[kD];
      tmem_ld128(tmem_base + (it & 1) * 256 + lane_addr, v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) tc2::mbar_arrive_leader(bar_d2_empty + 8 * (it & 1));
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int c = 0; c < kD; c += 4) { s0 += v[c]; s1 += v[c + 1]; s2 += v[c + 2]; s3 += v[c + 3]; }
      const float mean = ((s0 + s1) + (s2 + s3)) * (1.f / kD);
      s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
      for (int c = 0; c < kD; c += 4) {
        const float d0 = v[c] - mean, d1 = v[c + 1] - mean, d2 = v[c + 2] - mean, d3 = v[c + 3] - mean;
        s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
      }
      const float rstd = rsqrtf(((s0 + s1) + (s2 + s3)) * (1.f / kD) + 1e-5f);
      const float4* g4 = reinterpret_cast<const float4*>(gamma);
      const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
      for (int c = 0; c < kD; c += 4) {
        const float4 g = __ldg(g4 + (c >> 2)), b = __ldg(b4 + (c >> 2));
        v[c] = fmaf((v[c] - mean) * rstd, g.x, b.x); v[c + 1] = fmaf((v[c + 1] - mean) * rstd, g.y, b.y);
        v[c + 2] = fmaf((v[c + 2] - mean) * rstd, g.z, b.z); v[c + 3] = fmaf((v[c + 3] - mean) * rstd, g.w, b.w);
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {                     // + x: residual rows through the staging box
        if (lane == 0) {
          tma_store_wait_read();
          mbar_expect_tx(bar_my_res, kStageOutBytes);
          tma_load_2d(stage_buf, &mapR, bar_my_res, half * 64, row0);
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
            v[half * 64 + c8 * 8 + 2 * e] += __uint_as_float(w[e] << 16);
            v[half * 64 + c8 * 8 + 2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
          }
        }
        __syncwarp();
      }
      const int T = kBounded ? *live_rows_smem : T_cap;
      const bool whole_box = !kBounded || row0 + 32 <= T || T == T_cap;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          const int c = half * 64 + c8 * 8;
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                       ::"r"(my_row + ((uint32_t(c8) ^ sw) << 4)), "r"(pack_bf16(v[c], v[c + 1])),
                         "r"(pack_bf16(v[c + 2], v[c + 3])), "r"(pack_bf16(v[c + 4], v[c + 5])),
                         "r"(pack_bf16(v[c + 6], v[c + 7])) : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (whole_box) {
          if (lane == 0) {
            tma_store_2d(&mapO, stage_buf, half * 64, row0);
            tma_store_commit();
          }
        } else {
          if (row0 + lane < T) store_staged_half_row(my_row, sw, out + size_t(row0 + lane) * kD + half * 64);
          __syncwarp();
        }
      }
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  tc2::cluster_sync_all();                                       // the peer may still be signalling / reading this CTA
  if (warp == 1) {
    tc_fence_after();
    tc2::tmem_dealloc(tmem_base, 512u);
  }
}

// ---- linear attention, one warp per 25-token window ------------------------------------------------------------------
// q, k already hold elu(.)+1 and v holds values / S (fused into the projection's epilogue).  Per head h (16 dims):
//   KV[d][e] = sum_s k[s][d] v[s][e],  ksum[d] = sum_s k[s][d],  out[l][e] = S * (q[l] . KV[:, e]) / (q[l] . ksum + eps)
// Phase 1: lane (h, r) accumulates KV rows d = 4r..4r+3 (64 values) over the window; the 256 values of a head go through
// shared memory so that in phase 2 lane (h, r) owns output columns e = 4r..4r+3 for every token (no shuffles).
constexpr int kAttnWarps = 4;

__global__ void __launch_bounds__(kAttnWarps * 32)
fine_attn_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k, const __nv_bfloat16* __restrict__ v,
                 __nv_bfloat16* __restrict__ out, int64_t m, const int32_t* live, int S, float eps) {
  __shared__ float kv_s[kAttnWarps][kHeads][kHeadDim][kHeadDim + 1];
  __shared__ float ks_s[kAttnWarps][kHeads][kHeadDim];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = lane >> 2, r = lane & 3;
  const int64_t w = int64_t(blockIdx.x) * kAttnWarps + warp;
  if (w >= live_count(m, live, 1)) return;
  const size_t base = size_t(w) * S * kD;
  float kv[4][kHeadDim], ks[4];
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    ks[d] = 0.f;
#pragma unroll
    for (int e = 0; e < kHeadDim; ++e) kv[d][e] = 0.f;
  }
  for (int s = 0; s < S; ++s) {
    const uint2 kk = *reinterpret_cast<const uint2*>(k + base + size_t(s) * kD + h * kHeadDim + 4 * r);
    const uint4* vp = reinterpret_cast<const uint4*>(v + base + size_t(s) * kD + h * kHeadDim);
    const uint4 v0 = vp[0], v1 = vp[1];
    const float kd[4] = {__uint_as_float(kk.x << 16), __uint_as_float(kk.x & 0xffff0000u), __uint_as_float(kk.y << 16),
                         __uint_as_float(kk.y & 0xffff0000u)};
    const uint32_t vw[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    float ve[kHeadDim];
#pragma unroll
    for (int e = 0; e < 8; ++e) { ve[2 * e] = __uint_as_float(vw[e] << 16); ve[2 * e + 1] = __uint_as_float(vw[e] & 0xffff0000u); }
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      ks[d] += kd[d];
#pragma unroll
      for (int e = 0; e < kHeadDim; ++e) kv[d][e] = fmaf(kd[d], ve[e], kv[d][e]);
    }
  }
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    ks_s[warp][h][4 * r + d] = ks[d];
#pragma unroll
    for (int e = 0; e < kHeadDim; ++e) kv_s[warp][h][4 * r + d][e] = kv[d][e];
  }
  __syncwarp();
  float kvc[kHeadDim][4], ksum[kHeadDim];       // KV[:, 4r..4r+3] and sum_s k of this head
#pragma unroll
  for (int d = 0; d < kHeadDim; ++d) {
    ksum[d] = ks_s[warp][h][d];
#pragma unroll
    for (int e = 0; e < 4; ++e) kvc[d][e] = kv_s[warp][h][d][4 * r + e];
  }
  const float fs = float(S);
  for (int l = 0; l < S; ++l) {
    const uint4* qp = reinterpret_cast<const uint4*>(q + base + size_t(l) * kD + h * kHeadDim);
    const uint4 q0 = qp[0], q1 = qp[1];
    const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    float z = 0.f, o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float qa = __uint_as_float(qw[e] << 16), qb = __uint_as_float(qw[e] & 0xffff0000u);
      z = fmaf(qa, ksum[2 * e], z);
      z = fmaf(qb, ksum[2 * e + 1], z);
#pragma unroll
      for (int c = 0; c < 4; ++c) o[c] = fmaf(qa, kvc[2 * e][c], fmaf(qb, kvc[2 * e + 1][c], o[c]));
    }
    const float zi = fs / (z + eps);
    *reinterpret_cast<uint2*>(out + base + size_t(l) * kD + h * kHeadDim + 4 * r) =
        make_uint2(pack_bf16(o[0] * zi, o[1] * zi), pack_bf16(o[2] * zi, o[3] * zi));
  }
}

// ---- linear attention on warp-level tensor-core MMAs (windows of at most 32 tokens) ---------------------------------------
// The per-head blocks are 16 x 16 with a 25-token contraction: far below the 64/128-row granularity of tcgen05, so this
// kernel uses mma.sync.m16n8k16 (bf16 in, fp32 accumulate), one warp per window:
//   tiles      q, k, v [32 x 128] bf16 arrive with cp.async (16 B per lane, coalesced) into XOR-swizzled shared memory;
//              rows S..31 stay zero
//   phase 1    per head: C' = V_h^T K_h (= KV^T, rows = value dim, cols = key dim) and, through a constant A fragment
//              whose row 0 is all ones, ksum = sum_s K_h[s]        (8 MMAs, operands via ldmatrix.trans)
//   phase 2    per head: out_h = Q_h KV_h; the accumulator fragment of C' IS the B fragment of KV (rounded to bf16);
//              z = q . ksum stays fp32 (partial dot on the A fragment + 2 shuffles); rows scaled by S / (z + eps)
//   output     staged in shared memory (padded pitch), written with coalesced 16-byte stores
constexpr int kMmaWarps = 4;
constexpr int kTileRows = 32, kTileBytes = kTileRows * kD * 2;          // 8 KB per tile
constexpr int kAttnSmemPerWarp = 3 * kTileBytes;
constexpr int kOutPitch = kD * 2 + 16;                                   // bytes; +16: conflict-free fragment stores

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// Phases 1 and 2 + store for ONE window whose q / k / v tiles ([32 x 128] bf16, XOR-swizzled rows of 256 B, rows S..31 zero in
// k and v) are in shared memory at sq / sk / sv.  The k tile is reused as the output staging area and its tail is cleared
// again afterwards.  `out`: the window's [S, 128] rows in global memory.
__device__ __forceinline__ void attn_window_core(uint32_t sq, uint32_t sk, uint32_t sv, int S, float eps,
                                                 __nv_bfloat16* __restrict__ out, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const int nchunk = S * (kD * 2 / 16);                     // 16-byte chunks of one [S, 128] tile
  const float fs = float(S);
  const uint32_t ones = (g == 0) ? 0x3f803f80u : 0u;        // A fragment of the "row 0 = all ones" matrix
  const int lrow = lane & 7, lmat = lane >> 3;              // ldmatrix: this lane addresses row lrow of matrix lmat
  const size_t base = 0;
  // ---- phase 1: per head KV^T (16 x 16) and ksum (16) in fp32 accumulators ---------------------------------------
  float kvt[kHeads][2][4];        // [head][key-dim tile][fragment]: rows = value dim (g, g+8), cols = key dim 2t, 2t+1
  float ksum[kHeads][4];          // ksum[16h + {2t, 2t+1, 2t+8, 2t+9}] (valid in lanes with g == 0, broadcast below)
#pragma unroll
  for (int h = 0; h < kHeads; ++h) {
    float one_acc[2][4];
#pragma unroll
    for (int n = 0; n < 2; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) { kvt[h][n][e] = 0.f; one_acc[n][e] = 0.f; }
#pragma unroll
    for (int s0 = 0; s0 < kTileRows; s0 += 16) {
      uint32_t a[4], b[4];
      {   // A = V_h^T: matrices (tokens s0.., chunk 2h), (s0.., 2h+1), (s0+8.., 2h), (s0+8.., 2h+1), transposed
        const int row = s0 + ((lmat >> 1) << 3) + lrow, chunk = 2 * h + (lmat & 1);
        ldsm_x4_trans(sv + uint32_t(row) * 256u + (uint32_t(chunk ^ (row & 7)) << 4), a);
      }
      {   // B = K_h: matrices (s0.., 2h), (s0+8.., 2h), (s0.., 2h+1), (s0+8.., 2h+1), transposed
        const int row = s0 + ((lmat & 1) << 3) + lrow, chunk = 2 * h + (lmat >> 1);
        ldsm_x4_trans(sk + uint32_t(row) * 256u + (uint32_t(chunk ^ (row & 7)) << 4), b);
      }
      mma_bf16(kvt[h][0], a[0], a[1], a[2], a[3], b[0], b[1]);
      mma_bf16(kvt[h][1], a[0], a[1], a[2], a[3], b[2], b[3]);
      mma_bf16(one_acc[0], ones, 0u, ones, 0u, b[0], b[1]);
      mma_bf16(one_acc[1], ones, 0u, ones, 0u, b[2], b[3]);
    }
    // row 0 of the ones-product lives in lanes g == 0: lane t holds key dims 2t, 2t+1 (tile 0) and 2t+8, 2t+9 (tile 1)
    ksum[h][0] = __shfl_sync(kFullMask, one_acc[0][0], t);
    ksum[h][1] = __shfl_sync(kFullMask, one_acc[0][1], t);
    ksum[h][2] = __shfl_sync(kFullMask, one_acc[1][0], t);
    ksum[h][3] = __shfl_sync(kFullMask, one_acc[1][1], t);
  }
  __syncwarp();                   // every lane is done reading the k tile: it becomes the output staging area

  // ---- phase 2: out_h = (Q_h KV_h) * S / (Q_h . ksum + eps) ------------------------------------------------------
#pragma unroll
  for (int h = 0; h < kHeads; ++h) {
    // B fragments of KV_h from the accumulators of KV_h^T: value-dim tile 0 <- rows g (c0, c1), tile 1 <- rows g+8
    const uint32_t b00 = pack_bf16(kvt[h][0][0], kvt[h][0][1]), b01 = pack_bf16(kvt[h][1][0], kvt[h][1][1]);
    const uint32_t b10 = pack_bf16(kvt[h][0][2], kvt[h][0][3]), b11 = pack_bf16(kvt[h][1][2], kvt[h][1][3]);
#pragma unroll
    for (int m0 = 0; m0 < kTileRows; m0 += 16) {
      if (m0 >= S) break;
      uint32_t a[4];
      {   // A = Q_h: matrices (tokens m0.., chunk 2h), (m0+8.., 2h), (m0.., 2h+1), (m0+8.., 2h+1)
        const int row = m0 + ((lmat & 1) << 3) + lrow, chunk = 2 * h + (lmat >> 1);
        ldsm_x4(sq + uint32_t(row) * 256u + (uint32_t(chunk ^ (row & 7)) << 4), a);
      }
      float o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};
      mma_bf16(o0, a[0], a[1], a[2], a[3], b00, b01);
      mma_bf16(o1, a[0], a[1], a[2], a[3], b10, b11);
      float z0 = bf_lo(a[0]) * ksum[h][0] + bf_hi(a[0]) * ksum[h][1] + bf_lo(a[2]) * ksum[h][2] + bf_hi(a[2]) * ksum[h][3];
      float z1 = bf_lo(a[1]) * ksum[h][0] + bf_hi(a[1]) * ksum[h][1] + bf_lo(a[3]) * ksum[h][2] + bf_hi(a[3]) * ksum[h][3];
      z0 += __shfl_xor_sync(kFullMask, z0, 1); z0 += __shfl_xor_sync(kFullMask, z0, 2);
      z1 += __shfl_xor_sync(kFullMask, z1, 1); z1 += __shfl_xor_sync(kFullMask, z1, 2);
      const float zi0 = fs / (z0 + eps), zi1 = fs / (z1 + eps);
      const uint32_t r0 = sk + uint32_t(m0 + g) * kOutPitch + uint32_t(16 * h + 2 * t) * 2;
      const uint32_t r1 = r0 + 8 * kOutPitch;
      if (m0 + g < S) {
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r0), "r"(pack_bf16(o0[0] * zi0, o0[1] * zi0)) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r0 + 16), "r"(pack_bf16(o1[0] * zi0, o1[1] * zi0)) : "memory");
      }
      if (m0 + g + 8 < S) {
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r1), "r"(pack_bf16(o0[2] * zi1, o0[3] * zi1)) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r1 + 16), "r"(pack_bf16(o1[2] * zi1, o1[3] * zi1)) : "memory");
      }
    }
  }
  __syncwarp();
  // ---- store: 16 bytes per lane, consecutive lanes -> consecutive addresses -------------------------------------------
  for (int i = lane; i < nchunk; i += 32) {
    const int r = i >> 4, c = i & 15;
    uint4 val;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                 : "r"(sk + uint32_t(r) * kOutPitch + uint32_t(c) * 16));
    *reinterpret_cast<uint4*>(out + base + size_t(i) * 8) = val;
  }
  __syncwarp();
  // the staging area overwrote rows of the k tile beyond what the next load rewrites (pitch 272 vs 256): clear the tail
  for (int i = lane; i < (kTileRows - S) * 16 + 16; i += 32) {
    const uint32_t off = uint32_t(kTileBytes) - 16u * uint32_t(i + 1);
    if (off >= uint32_t(S) * 256u) asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(sk + off), "r"(0u) : "memory");
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kMmaWarps * 32)
fine_attn_mma_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                     const __nv_bfloat16* __restrict__ v, __nv_bfloat16* __restrict__ out, int64_t m, const int32_t* live,
                     int S, float eps) {
  extern __shared__ __align__(128) uint8_t attn_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const uint32_t sq = smem_u32(attn_smem) + warp * kAttnSmemPerWarp, sk = sq + kTileBytes, sv = sk + kTileBytes;
  // zero the three tiles once: rows S..31 are never written again
  for (int i = lane; i < kAttnSmemPerWarp / 16; i += 32)
    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(sq + i * 16), "r"(0u) : "memory");
  __syncwarp();
  const int nchunk = S * (kD * 2 / 16);                     // 16-byte chunks of one [S, 128] tile
  const int64_t m_live = live_count(m, live, 1);

  for (int64_t w = int64_t(blockIdx.x) * kMmaWarps + warp; w < m_live; w += int64_t(gridDim.x) * kMmaWarps) {
    const size_t base = size_t(w) * S * kD;
    // ---- load: chunk c of row r lands at r * 256 + ((c ^ (r & 7)) << 4) --------------------------------------------
    for (int i = lane; i < nchunk; i += 32) {
      const int r = i >> 4, c = i & 15;
      const uint32_t off = uint32_t(r) * 256u + (uint32_t(c ^ (r & 7)) << 4);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sk + off), "l"(k + base + size_t(i) * 8) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sv + off), "l"(v + base + size_t(i) * 8) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sq + off), "l"(q + base + size_t(i) * 8) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    __syncwarp();

    attn_window_core(sq, sk, sv, S, eps, out + base, lane);
  }
}

// rows [0, m): f0[b, i, :], rows [m, 2m): f1[b, j, :]   (fine_preprocess.py:50-51, the cat along dim 0); with a live count
// only rows [0, live) and [m, m + live) (the ids past it are never read)
__global__ void __launch_bounds__(256) gather_coarse_rows_kernel(const __nv_bfloat16* __restrict__ f0,
                                                                const __nv_bfloat16* __restrict__ f1,
                                                                const int64_t* __restrict__ b_ids,
                                                                const int64_t* __restrict__ i_ids,
                                                                const int64_t* __restrict__ j_ids, int64_t m,
                                                                const int32_t* __restrict__ live, int L, int S, int C,
                                                                __nv_bfloat16* __restrict__ out) {
  const int64_t row = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= 2 * m) return;
  const int lane = threadIdx.x & 31;
  const bool second = row >= m;
  const int64_t mm = second ? row - m : row;
  if (mm >= live_count(m, live, 1)) return;
  const __nv_bfloat16* src = second ? f1 + (size_t(b_ids[mm]) * S + size_t(j_ids[mm])) * C
                                    : f0 + (size_t(b_ids[mm]) * L + size_t(i_ids[mm])) * C;
  for (int c = lane * 8; c < C; c += 256)
    *reinterpret_cast<uint4*>(out + size_t(row) * C + c) = *reinterpret_cast<const uint4*>(src + c);
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct Dst { void* ptr; int64_t pitch; };                   // one 128-column block of the output (bf16, row pitch in elements)

// Y[T, N] = epilogue(X[T, K] . W[N, K]^T), X contiguous bf16;  out[j] receives output columns [128 j, 128 j + 128).
// live (may be null): device count of live items of rows_per_item rows each; T is then the capacity.
cudaError_t linear_run(int64_t T, const int32_t* live, int rows_per_item, const void* X, const void* W, int N, int K,
                       int64_t w_pitch, const Dst (&out)[3], LinParams P, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (T > 0x7fffffff - kTile || N % 128 || K % kBoxK || (N / 128) * (K / kBoxK) > kMaxWBoxes || N / 128 > 3)
    return cudaErrorInvalidValue;
  CUtensorMap mx, mw, mo[3];
  if (!make_map2d(&mx, X, T, K, K)) return cudaErrorInvalidValue;
  if (!make_map2d(&mw, W, N, K, w_pitch)) return cudaErrorInvalidValue;
  const void* any_out = P.out_f32 ? X : out[0].ptr;            // unused maps still have to be valid descriptors
  for (int j = 0; j < 3; ++j) {
    const bool used = !P.out_f32 && j < N / 128;
    if (used && !out[j].ptr) return cudaErrorInvalidValue;
    if (!make_map2d(&mo[j], used ? out[j].ptr : any_out, T, kD, used ? out[j].pitch : kD, 32)) return cudaErrorInvalidValue;
    P.out_rows[j] = used ? static_cast<__nv_bfloat16*>(out[j].ptr) : nullptr;
    P.out_pitch[j] = used ? int(out[j].pitch) : 0;
  }
  P.T = int(T);
  P.live = live;
  P.rows_per_item = rows_per_item;
  P.kchunks = K / kBoxK;
  P.nblk = N / 128;
  P.stages = min(kMaxStages, (kSmemBudget - 1024 - kSmemW - P.nblk * P.kchunks * kBoxBytes) / kBoxBytes);
  if (P.stages < 2) return cudaErrorInvalidValue;
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  const auto kernel = live ? linear_tc_kernel<true> : linear_tc_kernel<false>;
  if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemAlloc)) != cudaSuccess) return e;
  const int ntiles = int((T + kTile - 1) / kTile);
  kernel<<<min(ntiles, sms), kLinThreads, kSmemAlloc, st>>>(mx, mw, mo[0], mo[1], mo[2], P);
  return cudaGetLastError();
}

// x <- x + LayerNorm(W2 . relu(W1 . cat(x, m1))) in place, one launch
cudaError_t mlp_fused_run(__nv_bfloat16* x, const __nv_bfloat16* m1, int64_t T, const int32_t* live, int rows_per_item,
                          const void* W1, const void* W2, const float* gamma, const float* beta, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (T > 0x7fffffff - 2 * kTile) return cudaErrorInvalidValue;
  CUtensorMap mx, mm, mw1, mw2, mo, mr;
  if (!make_map2d(&mx, x, T, kD, kD) || !make_map2d(&mm, m1, T, kD, kD) || !make_map2d(&mw1, W1, 256, 256, 256) ||
      !make_map2d(&mw2, W2, 128, 256, 256, 64) || !make_map2d(&mo, x, T, kD, kD, 32) || !make_map2d(&mr, x, T, kD, kD, 32))
    return cudaErrorInvalidValue;
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  const auto kernel = live ? mlp_fused_kernel<true> : mlp_fused_kernel<false>;
  if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fm::kFmAlloc)) != cudaSuccess) return e;
  const int ntiles = int((T + 2 * kTile - 1) / (2 * kTile));
  kernel<<<2 * min(ntiles, sms / 2), fm::kFmThreads, fm::kFmAlloc, st>>>(mx, mm, mw1, mw2, mo, mr, int(T), live, rows_per_item, x,
                                                                         gamma, beta);
  return cudaGetLastError();
}

// packed weights of one LoFTREncoderLayer (byte offsets; matrices bf16 row-major [out, in] like nn.Linear.weight)
constexpr size_t kOffQkv = 0;                                  // [384, 128]  q_proj, k_proj, v_proj stacked
constexpr size_t kOffMerge = kOffQkv + 384 * 128 * 2;          // [128, 128]
constexpr size_t kOffMlp1 = kOffMerge + 128 * 128 * 2;         // [256, 256]
constexpr size_t kOffMlp2 = kOffMlp1 + 256 * 256 * 2;          // [128, 256]
constexpr size_t kOffLn = kOffMlp2 + 128 * 256 * 2;            // fp32: norm1.weight, norm1.bias, norm2.weight, norm2.bias
constexpr size_t kLayerBytes = kOffLn + 4 * 128 * 4;
static_assert(kLayerBytes == POPE_FINE_TF_LAYER_BYTES, "include/pope_b200.h documents this layout");
// FinePreprocess Linears
constexpr size_t kOffDown = 0;                                 // down_proj.weight [128, 256]
constexpr size_t kOffMergeFeat = kOffDown + 128 * 256 * 2;     // merge_feat.weight [128, 256]
constexpr size_t kOffPreBias = kOffMergeFeat + 128 * 256 * 2;  // fp32: down_proj.bias [128], merge_feat.bias [128]
constexpr size_t kPreBytes = kOffPreBias + 2 * 128 * 4;
static_assert(kPreBytes == POPE_FINE_PRE_BYTES, "include/pope_b200.h documents this layout");

struct TfScratch { __nv_bfloat16 *q, *k, *v, *msg, *m1; size_t bytes; };
TfScratch carve_tf(void* base, int64_t m, int S) {
  TfScratch w;
  char* p = static_cast<char*>(base);
  const size_t unit = align_up(size_t(m) * S * kD * 2, 256);
  size_t off = 0;
  w.q = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.k = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.v = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.msg = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.m1 = reinterpret_cast<__nv_bfloat16*>(p + off); off += unit;
  w.bytes = off;
  return w;
}

cudaError_t attention_run(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* v, __nv_bfloat16* out, int64_t m,
                          const int32_t* live, int S, cudaStream_t st) {
  if (S > kTileRows) {
    fine_attn_kernel<<<unsigned((m + kAttnWarps - 1) / kAttnWarps), kAttnWarps * 32, 0, st>>>(q, k, v, out, m, live, S, 1e-6f);
    return cudaGetLastError();
  }
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  constexpr int smem = kMmaWarps * kAttnSmemPerWarp;
  if ((e = cudaFuncSetAttribute(fine_attn_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return e;
  const int64_t blocks = (m + kMmaWarps - 1) / kMmaWarps;
  fine_attn_mma_kernel<<<unsigned(blocks < int64_t(sms) * 2 ? blocks : int64_t(sms) * 2), kMmaWarps * 32, smem, st>>>(q, k, v, out, m,
                                                                                                                 live, S, 1e-6f);
  return cudaGetLastError();
}

// x <- x + norm2(mlp(cat(x, norm1(merge(attention(q(x), k(src), v(src)))))))      (transformer.py:34-58), in place on x
cudaError_t encoder_layer(__nv_bfloat16* x, const __nv_bfloat16* src, int64_t m, const int32_t* live, int S, const char* wl,
                          const TfScratch& w, cudaStream_t st) {
  const int64_t T = m * S;
  const float* ln = reinterpret_cast<const float*>(wl + kOffLn);
  cudaError_t e;
  LinParams P{};
  if (x == src) {                       // self: one pass over x produces q, k, v
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_ELU1; P.mode[2] = EPI_SCALE; P.scale = 1.f / float(S);
    const Dst o[3] = {{w.q, kD}, {w.k, kD}, {w.v, kD}};
    if ((e = linear_run(T, live, S, x, wl + kOffQkv, 384, kD, kD, o, P, st)) != cudaSuccess) return e;
  } else {
    P.mode[0] = EPI_ELU1;
    const Dst oq[3] = {{w.q, kD}, {nullptr, 0}, {nullptr, 0}};
    if ((e = linear_run(T, live, S, x, wl + kOffQkv, 128, kD, kD, oq, P, st)) != cudaSuccess) return e;
    P.mode[0] = EPI_ELU1; P.mode[1] = EPI_SCALE; P.scale = 1.f / float(S);
    const Dst okv[3] = {{w.k, kD}, {w.v, kD}, {nullptr, 0}};
    if ((e = linear_run(T, live, S, src, wl + kOffQkv + 128 * 128 * 2, 256, kD, kD, okv, P, st)) != cudaSuccess) return e;
  }
  if ((e = attention_run(w.q, w.k, w.v, w.msg, m, live, S, st)) != cudaSuccess) return e;
  P = LinParams{};
  P.mode[0] = EPI_LN; P.gamma = ln; P.beta = ln + 128;
  const Dst om[3] = {{w.m1, kD}, {nullptr, 0}, {nullptr, 0}};
  if ((e = linear_run(T, live, S, w.msg, wl + kOffMerge, 128, kD, kD, om, P, st)) != cudaSuccess) return e;
  return mlp_fused_run(x, w.m1, T, live, S, wl + kOffMlp1, wl + kOffMlp2, ln + 256, ln + 384, st);
}

}  // namespace
}  // namespace pope

using namespace pope;

extern "C" size_t pope_fine_tf_workspace_bytes(int64_t m_windows, int window_tokens) {
  if (m_windows <= 0 || window_tokens <= 0) return 0;
  return carve_tf(nullptr, m_windows, window_tokens).bytes;
}

extern "C" int pope_fine_transformer_ex(void* feat0, void* feat1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                                        const void* weights, int n_layers, const int* layer_kinds, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  if (!feat0 || !feat1 || !weights || !layer_kinds || !workspace) return POPE_ERR_INVALID_ARG;
  if (m_windows < 0 || window_tokens <= 0 || n_layers < 0) return POPE_ERR_INVALID_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (layer_kinds[l] != 0 && layer_kinds[l] != 1) return POPE_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(feat0) | reinterpret_cast<uintptr_t>(feat1) | reinterpret_cast<uintptr_t>(weights) |
       reinterpret_cast<uintptr_t>(workspace)) & 15u)
    return POPE_ERR_ALIGNMENT;
  if (m_windows == 0) return POPE_OK;
  const TfScratch w = carve_tf(workspace, m_windows, window_tokens);
  if (workspace_bytes < w.bytes) return POPE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* x0 = static_cast<__nv_bfloat16*>(feat0);
  __nv_bfloat16* x1 = static_cast<__nv_bfloat16*>(feat1);
  for (int l = 0; l < n_layers; ++l) {
    const char* wl = static_cast<const char*>(weights) + size_t(l) * kLayerBytes;
    cudaError_t e;
    if (layer_kinds[l] == 0) {            // 'self'  (transformer.py:96-98)
      if ((e = encoder_layer(x0, x0, m_windows, m_dev, window_tokens, wl, w, st)) != cudaSuccess) return int(e);
      if ((e = encoder_layer(x1, x1, m_windows, m_dev, window_tokens, wl, w, st)) != cudaSuccess) return int(e);
    } else {                              // 'cross' (:99-101): feat1 attends to the UPDATED feat0
      if ((e = encoder_layer(x0, x1, m_windows, m_dev, window_tokens, wl, w, st)) != cudaSuccess) return int(e);
      if ((e = encoder_layer(x1, x0, m_windows, m_dev, window_tokens, wl, w, st)) != cudaSuccess) return int(e);
    }
  }
  return POPE_OK;
}

extern "C" int pope_fine_transformer(void* feat0, void* feat1, int64_t m_windows, int window_tokens, const void* weights,
                                     int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  return pope_fine_transformer_ex(feat0, feat1, m_windows, nullptr, window_tokens, weights, n_layers, layer_kinds, workspace,
                                  workspace_bytes, stream);
}

static size_t merge_scratch_bytes(int64_t m) {
  // gathered coarse rows [2m, 256] bf16, projected rows [2m, 128] bf16, per-window vectors [2m, 128] fp32
  return align_up(size_t(2 * m) * 256 * 2, 256) + align_up(size_t(2 * m) * 128 * 2, 256) + align_up(size_t(2 * m) * 128 * 4, 256);
}

extern "C" size_t pope_fine_merge_workspace_bytes(int64_t m_windows) {
  return m_windows > 0 ? merge_scratch_bytes(m_windows) : 0;
}

extern "C" int pope_fine_merge_coarse_ex(void* win0, void* win1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                                         const void* feat_c0, const void* feat_c1, int L, int S, int C, const int64_t* b_ids,
                                         const int64_t* i_ids, const int64_t* j_ids, const void* weights, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  if (!win0 || !win1 || !feat_c0 || !feat_c1 || !b_ids || !i_ids || !j_ids || !weights || !workspace)
    return POPE_ERR_INVALID_ARG;
  if (m_windows < 0 || window_tokens <= 0 || L <= 0 || S <= 0) return POPE_ERR_INVALID_ARG;
  if (C != 256) return POPE_ERR_SHAPE;
  if (m_windows == 0) return POPE_OK;
  if (workspace_bytes < merge_scratch_bytes(m_windows)) return POPE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t m = m_windows;
  char* p = static_cast<char*>(workspace);
  __nv_bfloat16* cg = reinterpret_cast<__nv_bfloat16*>(p);
  __nv_bfloat16* cd = reinterpret_cast<__nv_bfloat16*>(p + align_up(size_t(2 * m) * 256 * 2, 256));
  float* cvec = reinterpret_cast<float*>(reinterpret_cast<char*>(cd) + align_up(size_t(2 * m) * 128 * 2, 256));
  const char* wp = static_cast<const char*>(weights);
  const float* bias = reinterpret_cast<const float*>(wp + kOffPreBias);
  gather_coarse_rows_kernel<<<unsigned((2 * m + 7) / 8), 256, 0, st>>>(
      static_cast<const __nv_bfloat16*>(feat_c0), static_cast<const __nv_bfloat16*>(feat_c1), b_ids, i_ids, j_ids, m, m_dev, L, S,
      C, cg);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return int(e);
  // The [2m, .] arrays hold side 1 from row m (the capacity) on, so with a live count their live rows are [0, live) and
  // [m, m + live): each side is then its own launch, bounded by the count.  Without one, both sides are a single launch.
  const int nseg = m_dev ? 2 : 1;
  const int64_t seg = 2 * m / nseg;
  LinParams P{};
  for (int s = 0; s < nseg; ++s) {
    // feat_c_win = down_proj(cat(c0, c1))                                                (fine_preprocess.py:50-51)
    P = LinParams{};
    P.mode[0] = EPI_COPY; P.bias = bias;
    const Dst od[3] = {{cd + s * seg * kD, kD}, {nullptr, 0}, {nullptr, 0}};
    if ((e = linear_run(seg, m_dev, 1, cg + s * seg * 256, wp + kOffDown, 128, 256, 256, od, P, st)) != cudaSuccess) return int(e);
    // merge_feat(cat(win, repeat(c))) = win . Wa^T + (c . Wb^T + bias): the second term once per window     (:52-55)
    P = LinParams{};
    P.out_f32 = cvec + s * seg * kD; P.mode[0] = EPI_COPY; P.bias = bias + 128;
    const Dst onone[3] = {{nullptr, 0}, {nullptr, 0}, {nullptr, 0}};
    if ((e = linear_run(seg, m_dev, 1, cd + s * seg * kD, wp + kOffMergeFeat + 128 * 2, 128, 128, 256, onone, P, st)) != cudaSuccess)
      return int(e);
  }
  for (int side = 0; side < 2; ++side) {
    void* win = side ? win1 : win0;
    P = LinParams{};
    P.mode[0] = EPI_ADDVEC; P.rowvec = cvec + size_t(side) * m * kD; P.rows_per_vec = window_tokens;
    const Dst ow[3] = {{win, kD}, {nullptr, 0}, {nullptr, 0}};
    if ((e = linear_run(m * window_tokens, m_dev, window_tokens, win, wp + kOffMergeFeat, 128, 128, 256, ow, P, st)) != cudaSuccess)
      return int(e);
  }
  return POPE_OK;
}

extern "C" int pope_fine_merge_coarse(void* win0, void* win1, int64_t m_windows, int window_tokens, const void* feat_c0,
                                      const void* feat_c1, int L, int S, int C, const int64_t* b_ids, const int64_t* i_ids,
                                      const int64_t* j_ids, const void* weights, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  return pope_fine_merge_coarse_ex(win0, win1, m_windows, nullptr, window_tokens, feat_c0, feat_c1, L, S, C, b_ids, i_ids, j_ids,
                                   weights, workspace, workspace_bytes, stream);
}
