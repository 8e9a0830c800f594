// coarse_tc.cu -- coarse matching on the 5th-gen tensor cores (tcgen05 + TMEM + TMA), bf16 features, fp32 accumulate.
//
// Replaces src/matcher/utils/coarse_matching.py:106-119 and :175-189 of the reference (einsum -> /T -> dual softmax
// -> threshold -> mutual max) without ever writing the L x S matrix.  Sweeps over S = f0 f1^T (log2 units):
//   single sweep (thr > 0.15, the default 0.2): one pass over the rows of S computes 2^(x - m) with a lazily raised integer
//                           shift m per epilogue warp (32 rows): row sums per thread, column sums through a shuffle reduction
//                           as per-32-row partial sums (+ the shift they were taken at) that a small kernel merges into the
//                           column log-sum-exp, and per-thread candidate lists (below).  Pairs whose sums lose precision
//                           (rows more than ~186 log2 units apart inside one 32-row group, inf / nan) are flagged one by one
//                           and redone by a gated launch of the two-sweep kernel.
//   two sweeps (one launch): row log-sum-exp of S and of S^T (= column log-sum-exp of S), online softmax per row.  While
//                           sweeping the rows of S every epilogue thread also lists, in private slots (no atomics), the
//                           cells that exceed thr x the RUNNING row sum -- a superset of the cells with p_row > thr, of
//                           which a row has fewer than 1/thr; a small kernel evaluates the listed cells once both
//                           log-sum-exps are known.
//   sweep 3 (thr <= 0.15)  : recompute S, t2 = log2 conf = (x - lse_r[i]) + (x - lse_c[j]); cells above log2(thr) update
//                           the best-candidate record of their row and column (rare 64-bit atomicMax)
//
// Kernel anatomy (persistent, one CTA PAIR per two SMs, cta_group::2, 640 threads per CTA):
//   work unit   = (direction, pair, 256-row block of the stationary operand "A"); CTA r of the pair keeps rows
//                 [128r, 128r+128) of the block (64 KB) in its shared memory for the whole unit while 256-row tiles of
//                 the streamed operand "B" pass through an 8-stage ring: per stage each CTA TMA-loads ITS half of the
//                 tile (128 rows x 64 k, 16 KB, 128B-swizzled).  One tcgen05.mma.cta_group::2 (M=256, N=256, K=16)
//                 reads A and half of B from each SM: 64 B/clk of shared-memory reads and 32 B/clk of L2 traffic per
//                 SM (a single-CTA M=128 x N=128 tile needs 128 B/clk of shared-memory reads, i.e. all of it).
//   warps 0-15  = epilogue (four whole warpgroups): four threads per row (64 of the tile's 256 columns each); tcgen05.ld 32
//                 columns at a time; single sweep: FMNMX3 guard + FFMA2 + MUFU.EX2 + packed adds per element, a 7-shuffle
//                 column reduction and a candidate pre-test per 32x32 block; two-sweep: online softmax (FMNMX + FFMA +
//                 MUFU.EX2 + FADD per element); three-sweep: candidate test (FADD + FSETP per element, one warp vote per block)
//   warp 16     = TMA producer (one elected lane, both CTAs; transaction bytes land on the leader's barrier)
//   warp 17     = TMEM allocator (both CTAs) + tcgen05.mma issuer (leader CTA, one elected lane); accumulators are
//                 128 lanes x 256 fp32 columns per CTA, double-buffered (2 x 256 = all 512 TMEM columns); commits are
//                 multicast to the barriers of both CTAs
//   warps 18-19 = idle (they complete the fifth warpgroup): setmaxnreg moves registers from that warpgroup (40 per thread)
//                 to the epilogue warpgroups (104 per thread; a 640-thread CTA starts at 96, where the single-sweep epilogue
//                 spilled and re-derived thread constants from SR_TID for every tile)
//   barriers    = a_full/a_empty (stationary block), b_full/b_empty[8] (ring), acc_full/acc_empty[2] (TMEM stages);
//                 *_full of the operands and acc_empty live in the leader CTA (the issuer waits on them)
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace pope {
namespace {

using namespace tc1;

constexpr int kStages = 8;              // B ring depth
constexpr int kBoxRows = 128;           // rows per TMA box = rows of A / of the B half held by one CTA
constexpr int kBoxK = 64;               // bf16 elements per 128-byte swizzle row
constexpr int kBoxBytes = kBoxRows * kBoxK * 2;      // 16384
constexpr int kUnitRows = 256;          // stationary rows per work unit (128 per CTA of the pair)
constexpr int kTileCols = 256;          // streamed rows per tile (= MMA N; 128 loaded by each CTA)
constexpr int kMaxKChunks = 4;          // C <= 256
constexpr int kEpiWarps = 16;           // epilogue warps (multiple of 4: one per TMEM lane quadrant and column group)
constexpr int kColGroups = kEpiWarps / 4;            // threads per row
constexpr int kChunks = (256 / 32) / kColGroups;     // 32-column chunks per thread and tile
constexpr int kSpan = kChunks * 32;                  // columns per thread and tile
static_assert(kColGroups == kListGroups, "one private candidate list per (row, column group) thread");
constexpr int kEpiThreads = kEpiWarps * 32;
// warps 0..15 = epilogue (four whole warpgroups), warp 16 = TMA producer, warp 17 = TMEM allocator + MMA issuer, warps 18-19 idle:
// the epilogue warpgroups and the producer / issuer warpgroup trade registers with setmaxnreg (a 640-thread CTA starts at 96
// per thread; the data-movement warps need a fraction of that, the epilogue is short of registers at 96)
constexpr int kWarpProducer = kEpiWarps, kWarpMma = kEpiWarps + 1;
constexpr int kThreads = kEpiThreads + 128;
constexpr int kRegsEpi = 112, kRegsAux = 32;
static_assert(16 * 32 * kRegsEpi + 4 * 32 * kRegsAux <= 640 * 96, "setmaxnreg would wait for registers the CTA does not own");   // 16 x 32 x 112 + 4 x 32 x 32 = 61 440 = the CTA's 640 x 96 registers (the pool is per CTA)
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kIdesc = tc2::idesc_bf16_m256(kTileCols);   // every MMA: M = 256 (128 rows per CTA), N = one tile

// dynamic shared memory layout (base aligned to 1024 B for the 128B swizzle); identical in both CTAs of a pair
constexpr int kSmemA = 0;                                            // 4 k-chunks x 16 KB
// then (offsets computed inside the kernel, they depend on MODE): the stationary block(s), the ring of kStages (MODE 4: 5)
// 16 KB boxes, 4 KB of staged per-column terms / list counters, 3 KB of row-sum merge space, the barriers, the TMEM pointer
constexpr int kSmemAlloc = 2 * kMaxKChunks * kBoxBytes + 5 * kBoxBytes + 2 * 2 * kTileCols * 4 + 3 * 128 * 8 + 256 + 16 + 1024;
static_assert(kSmemAlloc >= kMaxKChunks * kBoxBytes + kStages * kBoxBytes + 2 * 2 * kTileCols * 4 + 3 * 128 * 8 + 256 + 16 + 1024 &&
              kSmemAlloc <= 227 * 1024, "shared-memory allocation");

struct SweepParams {
  // direction d: stationary operand = feature set d (rows LA[d]), streamed operand = the other one
  int n;                    // pairs covered by this launch ...
  int n_base;               // ... starting at this pair
  int L0, L1;               // rows of feature set 0 / 1; direction d has LA = L_d, LB = L_(1-d)
  int kchunks;
  int units_dir0;           // work units of direction 0 (direction 1 follows)
  int total_units;
  float scale_log2;
  float log2_thr;
  float* lse_out0;          // sweep 1+2: where direction 0 / 1 writes its row log-sum-exp
  float* lse_out1;
  const float* lse_r;       // sweep 3
  const float* lse_c;
  u64* rowbest;
  u64* colbest;
  int* cand_cnt;            // two-sweep path: per row of S, one count byte per column quarter
  u64* cand;                //   [n, L0, kListGroups, kListStride] (similarity in log2 units, float bits << 32 | column)
  float* colpart;           // single-sweep path: [n, ceil(L0/32), L1] column sums of 2^(x - shift) over each 32-row group
  float* cshift;            //   [n, ceil(L0/32), ceil(L1/32)] the shift of each (32-row group, 32-column block)
  int* pairflag;            //   [n] != 0: the pair left the single sweep's range and is redone by the gated launch
  int gate;                 // != 0: the launch is a no-op unless POPE_FLAG_ROBUST_PATH is set in *flags, and then only
                            //       the pairs with pairflag[n] != 0 are swept
  int32_t* flags;
};

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ void red_max_shared(uint32_t addr, int v) {
  asm volatile("red.shared.max.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float r;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr));
  return r;
}
__device__ __forceinline__ float tmem_ld1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n\ttcgen05.wait::ld.sync.aligned;" : "=r"(r) : "r"(taddr) : "memory");
  return __uint_as_float(r);
}

// online log-sum-exp update of one row with 32 more raw accumulators (vc of them valid)
__device__ __forceinline__ float lse_update(const float (&v)[32], int vc, float scale, float& m_run, float& s_run) {
  float cmax;
  if (vc >= 32) {
    float q0 = v[0], q1 = v[1], q2 = v[2], q3 = v[3];
#pragma unroll
    for (int j = 4; j < 32; j += 4) {
      q0 = fmaxf(q0, v[j]); q1 = fmaxf(q1, v[j + 1]); q2 = fmaxf(q2, v[j + 2]); q3 = fmaxf(q3, v[j + 3]);
    }
    cmax = fmaxf(fmaxf(q0, q1), fmaxf(q2, q3));
  } else {
    cmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) cmax = (j < vc) ? fmaxf(cmax, v[j]) : cmax;
  }
  const float m_new = fmaxf(m_run, cmax * scale);
  const float neg = -m_new;
  float a0 = s_run * ex2_approx(m_run - m_new), a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (vc >= 32) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      a0 += ex2_approx(fmaf(v[j + 0], scale, neg));
      a1 += ex2_approx(fmaf(v[j + 1], scale, neg));
      a2 += ex2_approx(fmaf(v[j + 2], scale, neg));
      a3 += ex2_approx(fmaf(v[j + 3], scale, neg));
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < vc) a1 += ex2_approx(fmaf(v[j], scale, neg));
  }
  s_run = (a0 + a1) + (a2 + a3);
  m_run = m_new;
  return cmax;      // raw-accumulator units
}

// append cell (similarity x in log2 units, column col) to one of the calling thread's private lists (SLOTS entries).  A full
// list is first re-filtered against the current bound (same units): the running row sum only grows, so entries below it
// are dead for good, and fewer than 1/thr cells can stay above it (heavy-tailed similarities list many early cells that a
// later, larger cell of the row makes irrelevant).  A list that is still full: two-sweep kernels raise
// POPE_FLAG_CAND_OVERFLOW (nan inputs), the single sweep hands the pair to the online-softmax launch.
template <int SLOTS>
__device__ __noinline__ int list_push(u64* __restrict__ list, int cnt, float bound, float v, int col, int32_t* __restrict__ flags,
                                      int* __restrict__ pairflag) {
  if (cnt >= SLOTS) {
    int kept = 0;
    for (int k = 0; k < SLOTS; ++k) {
      const u64 rec = list[k];
      if (__uint_as_float(uint32_t(rec >> 32)) > bound) list[kept++] = rec;
    }
    cnt = kept;
    if (cnt >= SLOTS) {
      if (pairflag) {
        atomicOr(reinterpret_cast<unsigned*>(flags), POPE_FLAG_ROBUST_PATH);
        *reinterpret_cast<volatile int*>(pairflag) = 1;
      } else {
        atomicOr(reinterpret_cast<unsigned*>(flags), POPE_FLAG_CAND_OVERFLOW);
      }
      return cnt;
    }
  }
  list[cnt] = (u64(__float_as_uint(v)) << 32) | uint32_t(col);
  return cnt + 1;
}

// ---- single-sweep path (MODE 3) ----------------------------------------------------------------------------------------
// Two tcgen05.ld.16x256b.x4 (lanes [0,16) and [16,32) of the warp's quadrant, 32 columns):
//   v[16h + 4k + 2r + c] = D[lane/4 + 8(2h + r)][8k + 2(lane%4) + c]      (checked on the device by tools/micro/tmem_layout.cu)
// so a thread holds 4 rows x 8 columns of the 32x32 block: row sums stay per thread, and a column sum needs 3 adds in
// the thread plus a 7-shuffle transposed reduction over the 8 lanes that share lane%4.
__device__ __forceinline__ void tmem_ld_frag(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%32];\n\t"
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%33];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr), "r"(taddr + (16u << 16)) : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// three-input maximum (sm_100 FMNMX3)
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// packed fp32x2 arithmetic (sm_100: one issue slot for two lanes of a 64-bit register pair)
__device__ __forceinline__ u64 pack2(float a, float b) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(u64 r, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(r)); }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
  u64 r;
  asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
  u64 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 r;
  asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// v <- e = 2^(v * scale - m) in place for the 32 raw accumulators of a thread (cells of ragged tiles that do not exist were
// set to -inf by the caller and come out as 0): all the multiply-adds can issue before the first exponential retires.  The
// (even, odd) column pairs of a row are adjacent registers, so scaling, the chunk's row sums (rc2[rho] = {even-column sum,
// odd-column sum}) and the per-thread column sums (cp2[k] = {column 8k+2p, column 8k+2p+1} over the thread's four rows) run
// on packed fp32x2 instructions
__device__ __forceinline__ void ss_chunk(float (&v)[32], float scale, float negm, u64 (&rc2)[4], u64 (&cp2)[4]) {
  const u64 scale2 = pack2(scale, scale), negm2 = pack2(negm, negm);
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int idx = 16 * h + 4 * k + 2 * r, rho = 2 * h + r;
        float a, b;
        unpack2(fma2(pack2(v[idx], v[idx + 1]), scale2, negm2), a, b);
        a = ex2_approx(a);
        b = ex2_approx(b);
        v[idx] = a;
        v[idx + 1] = b;
        const u64 e2 = pack2(a, b);
        rc2[rho] = (k == 0) ? e2 : add2(rc2[rho], e2);
        cp2[k] = (rho == 0) ? e2 : add2(cp2[k], e2);
      }
}

// ragged tiles: the cells of rows / columns that do not exist become -inf (2^-inf = 0 in every sum; no effect on the
// maximum that guards the shift).  Runs for the last tile / unit of a pair only.
__device__ __forceinline__ void ss_mask(float (&v)[32], uint32_t rowmask, int vc, int p) {
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int idx = 16 * h + 4 * k + 2 * r, rho = 2 * h + r;
        const int col = 8 * k + 2 * p;
        const bool rowok = (rowmask >> rho) & 1u;
        if (!rowok || col >= vc) v[idx] = -INFINITY;
        if (!rowok || col + 1 >= vc) v[idx + 1] = -INFINITY;
      }
}

// log2 of a positive normal float: exponent exactly, mantissa through lg2.approx (absolute error 2^-22)
__device__ __forceinline__ float log2_split(float e) {
  const uint32_t b = __float_as_uint(e);
  return float(int(b >> 23) - 127) + lg2_approx(__uint_as_float((b & 0x007fffffu) | 0x3f800000u));
}

// the 8 cells of one row of a chunk (e = 2^(x - m)) against the row's bound; cells above it go to the thread's private list
// as similarities in log2 units, x = log2(e) + m.  Returns the list's new fill count.  Out of line on purpose: the epilogue's
// hot loop must stay inside the instruction cache (64 KB of code cost 30 % of the kernel's time).
__device__ __noinline__ int ss_scan_row(float e0, float e1, float e2, float e3, float e4, float e5, float e6, float e7, float bound,
                                        float mshift, u64* __restrict__ list, int cnt, int col, int32_t* __restrict__ flags,
                                        int* __restrict__ pairflag) {
  // the bound a full list is re-filtered with, same units as the entries (margin on the safe side: the lists are a
  // superset anyway)
  const float xb = lg2_approx(bound) + mshift - 0.01f;
  const float e[8] = {e0, e1, e2, e3, e4, e5, e6, e7};
#pragma unroll
  for (int q = 0; q < 8; ++q)       // cell q: column col + 8 (q / 2) + q % 2
    if (e[q] > bound) cnt = list_push<kLaneSlots>(list, cnt, xb, log2_split(e[q]) + mshift, col + 8 * (q >> 1) + (q & 1), flags, pairflag);
  return cnt;
}

// transposed reduction of the 8 per-thread column sums over the 8 lanes with the same lane%4: lane l ends up with the
// sum of column c8 = l / 4 (chunk column 8(c8/2) + 2(l%4) + c8%2) over the warp's 32 rows; fixed order -> deterministic
__device__ __forceinline__ float ss_col_reduce(const float (&cp)[8], int lane) {
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  float q4[4], q2[2];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const float send = b4 ? cp[m] : cp[m + 4], keep = b4 ? cp[m + 4] : cp[m];
    q4[m] = keep + __shfl_xor_sync(kFullMask, send, 16);
  }
#pragma unroll
  for (int m = 0; m < 2; ++m) {
    const float send = b3 ? q4[m] : q4[m + 2], keep = b3 ? q4[m + 2] : q4[m];
    q2[m] = keep + __shfl_xor_sync(kFullMask, send, 8);
  }
  const float send = b2 ? q2[0] : q2[1], keep = b2 ? q2[1] : q2[0];
  return keep + __shfl_xor_sync(kFullMask, send, 4);
}

// MODE 0: row log-sum-exp of the stationary operand's rows.
// MODE 1: candidate sweep of the three-sweep path (needs both log-sum-exps; direction 0 only).
// MODE 2: MODE 0 + in direction 0 (rows of S stationary) every thread lists the cells of its row that exceed thr x the
//         running row sum in its private slots (two-sweep path; both directions run in one launch).
// MODE 3: single sweep over the rows of S (direction 0 only): 2^(x - m) with one lazily raised shift m per epilogue warp
//         (32 rows), row sums per thread, column sums through a shuffle reduction and per-32-row partial sums (plus the
//         shift they were taken at) in global memory, candidate lists as in MODE 2.  A pair whose sums lose precision
//         (rows more than ~150 log2 units apart inside one 32-row group, inf / nan) raises POPE_FLAG_ROBUST_PATH and its
//         own flag, and a gated MODE 2 launch redoes that pair.
// MODE 4: MODE 3 for FP32 features at fp32 accuracy on the bf16 tensor cores.  Every feature value is split into three bf16
//         terms a = a1 + a2 + a3 (24 mantissa bits, split3_kernel) and the contraction is the six significant products
//         a1b1 + a2b1 + a3b1 + a1b2 + a2b2 + a1b3 (the dropped ones are below 2^-24 of |a||b|) accumulated in fp32 in
//         TMEM -- 6x the MMAs of MODE 3, which hides the epilogue completely.  The a1 and a2 blocks of the unit stay
//         resident (128 KB), a3 and the b planes stream through a 5-stage ring.  maps: map0..2 = planes of f0,
//         map3..5 = planes of f1.
template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
sweep_tc_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1,
                const __grid_constant__ CUtensorMap map2, const __grid_constant__ CUtensorMap map3,
                const __grid_constant__ CUtensorMap map4, const __grid_constant__ CUtensorMap map5, const SweepParams P) {
  // shared-memory layout: MODE 4 keeps two stationary blocks (a1, a2) and a shorter ring
  constexpr int kAChunks = (MODE == 4) ? 2 * kMaxKChunks : kMaxKChunks;
  constexpr int kRing = (MODE == 4) ? 5 : kStages;
  constexpr int kSmemB = kSmemA + kAChunks * kBoxBytes;
  constexpr int kSmemLc = kSmemB + kRing * kBoxBytes;
  constexpr int kSmemMerge = kSmemLc + 2 * 2 * kTileCols * 4;
  constexpr int kSmemBar = kSmemMerge + 3 * 128 * 8;
  constexpr int kSmemTmemPtr = kSmemBar + (2 * kMaxKChunks + 2 * kRing + 4) * 8;
  static_assert(kSmemTmemPtr + 16 + 1024 <= kSmemAlloc, "shared-memory layout exceeds the allocation");
  constexpr int kStages = kRing;                    // shadows the file-level ring depth inside the kernel
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // (made opaque: otherwise the compiler re-derives the aligned shared-memory base -- S2UR SR_CgaCtaId and ~20 dependent
  //  instructions -- for every tile in the epilogue instead of spending a register on it)
  uint32_t sbase_pin = smem_u32(smem);
  asm volatile("" : "+r"(sbase_pin));
  const uint32_t sbase = sbase_pin;
  const uint32_t bar0 = sbase + kSmemBar;
  // one full / empty pair per 64-wide k-chunk of the stationary block: a chunk is reloaded for the next unit as soon as the
  // unit's LAST tile has read it, while the MMAs of the remaining chunks still run (the reload of the whole block after the
  // unit's last MMA used to cost about one tile time in twenty)
  const uint32_t bar_a_full = bar0, bar_a_empty = bar0 + 8 * kMaxKChunks;
  const uint32_t bar_b_full = bar0 + 16 * kMaxKChunks, bar_b_empty = bar_b_full + 8 * kStages;
  const uint32_t bar_acc_full = bar_b_empty + 8 * kStages, bar_acc_empty = bar_acc_full + 16;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kSmemTmemPtr);

  // (a kernel launched behind this one WITH programmatic stream serialisation may start while this one runs: the column
  //  merge of the head of a split single sweep, single_sweep_run; ordinary launches are not affected)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (P.gate && !(uint32_t(*reinterpret_cast<const volatile int32_t*>(P.flags)) & POPE_FLAG_ROBUST_PATH)) return;
  // (volatile read: the compiler otherwise re-derives lane bits from SR_TID.X inside the epilogue loops, ~6 S2R per chunk)
  uint32_t lane_u;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane_u));
  const int warp = threadIdx.x >> 5, lane = int(lane_u);
  const uint32_t rank = tc2::cluster_ctarank();     // 0 = leader (issues the MMAs), 1 = peer
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == kWarpProducer && lane == 0) {
    prefetch_tmap(&map0);
    prefetch_tmap(&map1);
    // operand "full" barriers: one arrival (the leader's expect_tx) + the bytes of both CTAs' TMA loads
    for (int b = 0; b < kMaxKChunks; ++b) {
      mbar_init(bar_a_full + 8 * b, 1);
      mbar_init(bar_a_empty + 8 * b, 1);             // one multicast tcgen05.commit
    }
    for (int s = 0; s < kStages; ++s) { mbar_init(bar_b_full + 8 * s, 1); mbar_init(bar_b_empty + 8 * s, 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);            // one multicast tcgen05.commit
      mbar_init(bar_acc_empty + 8 * s, 2 * kEpiWarps);   // one arrival per epilogue warp of BOTH CTAs (leader's copy)
    }
    fence_barrier_init();
  }
  if (warp == kWarpMma) {
    tc2::tmem_alloc(sbase + kSmemTmemPtr, kTmemCols);
    tc2::tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc2::cluster_sync_all();                           // peer barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int kchunks = P.kchunks;

  // unit -> (direction, pair, row block)
  auto decode = [&](int u, int& dir, int& n, int& rb) {
    dir = (u >= P.units_dir0) ? 1 : 0;
    const int v = dir ? u - P.units_dir0 : u;
    const int rbs = ((dir ? P.L1 : P.L0) + kUnitRows - 1) / kUnitRows;
    const int q = v / rbs;
    rb = v - q * rbs;
    n = P.n_base + q;          // (a launch may cover the pairs [n_base, n_base + n) only)
  };

  // gated launch (the fallback behind the single sweep): only the pairs the single sweep gave up on are swept; the
  // flags are final before this launch starts, so all roles of both CTAs skip the same units
  auto skip_pair = [&](int n) { return MODE == 2 && P.gate && *reinterpret_cast<const volatile int*>(P.pairflag + n) == 0; };

  if (warp >= kEpiWarps) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsAux));
  if (warp == kWarpProducer) {
    // =============================== TMA producer of the streamed operand (both CTAs) ===============================
    if (lane == 0) {
      uint32_t b_stage = 0, b_phase = 0;
      for (int u = pair; u < P.total_units; u += npairs) {
        int dir, n, rb;
        decode(u, dir, n, rb);
        if (skip_pair(n)) continue;
        const CUtensorMap* mapB = dir ? &map0 : &map1;
        const int arow = rb * kUnitRows + int(rank) * kBoxRows;
        auto ring_load = [&](const CUtensorMap* mp, int kc, int row) {
          mbar_wait_batched(bar_b_empty + 8 * b_stage, b_phase ^ 1);
          if (rank == 0) mbar_expect_tx(bar_b_full + 8 * b_stage, 2 * kBoxBytes);
          tc2::tma_load_3d_2sm(sbase + kSmemB + b_stage * kBoxBytes, mp, bar_b_full + 8 * b_stage, kc * kBoxK, row, n);
          if (++b_stage == kStages) { b_stage = 0; b_phase ^= 1; }
        };
        const int ntiles = ((dir ? P.L0 : P.L1) + kTileCols - 1) / kTileCols;
        for (int ct = 0; ct < ntiles; ++ct) {
          const int brow = ct * kTileCols + int(rank) * kBoxRows;
          if (MODE == 4) {
            // ring order = the issuer's order: (a3[c], b1[c]) for every k-chunk, then the b2 chunks, then the b3 chunks
            for (int kc = 0; kc < kchunks; ++kc) { ring_load(&map2, kc, arow); ring_load(&map3, kc, brow); }
            for (int kc = 0; kc < kchunks; ++kc) ring_load(&map4, kc, brow);
            for (int kc = 0; kc < kchunks; ++kc) ring_load(&map5, kc, brow);
          } else {
            for (int kc = 0; kc < kchunks; ++kc) ring_load(mapB, kc, brow);
          }
        }
      }
    }
  } else if (warp == kWarpMma) {
    // =============================== MMA issuer (leader CTA only) ===============================
    // The whole warp walks the loops (so that every counter and address is warp-uniform and stays in uniform registers:
    // with a single lane inside, the descriptors went through five R2UR broadcasts per MMA and a k-chunk took 130 clk
    // longer to issue); lane 0 alone issues the tcgen05 instructions.
    if (rank == 0) {
      uint32_t a_phase = 0, b_stage = 0, b_phase = 0, tile_ctr = 0;
      for (int u = pair; u < P.total_units; u += npairs) {
        int dir, n, rb;
        decode(u, dir, n, rb);
        if (skip_pair(n)) continue;
        const int ntiles = ((dir ? P.L0 : P.L1) + kTileCols - 1) / kTileCols;
        // k-chunk kc of the stationary block: awaited before its first use in the unit's first tile, handed back to the
        // loader right after its last use in the unit's last tile
        auto a_wait = [&](int ct, int kc) {
          if (ct == 0) { mbar_wait_batched(bar_a_full + 8 * kc, a_phase); tc_fence_after(); }
        };
        auto a_done = [&](int ct, int kc) {
          if (ct == ntiles - 1 && elect_one()) tc2::umma_commit(bar_a_empty + 8 * kc);
        };
        for (int ct = 0; ct < ntiles; ++ct, ++tile_ctr) {
          const uint32_t s = tile_ctr & 1, acc_phase = (tile_ctr >> 1) & 1;
          mbar_wait_batched(bar_acc_empty + 8 * s, acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d = tmem_base + s * kTileCols;
          if (MODE == 4) {
            // six products per k-chunk: (a1 + a2 + a3) b1, (a1 + a2) b2, a1 b3; a1 / a2 resident, a3 and b* from the ring
            uint32_t first = 0;
            auto mma4 = [&](uint32_t a_addr, uint32_t b_addr) {
              if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < kBoxK / 16; ++ks) tc2::umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), kIdesc, first | uint32_t(ks));
              }
              first = 1u;
            };
            auto ring_wait = [&]() {
              mbar_wait_batched(bar_b_full + 8 * b_stage, b_phase);
              tc_fence_after();
              const uint32_t addr = sbase + kSmemB + b_stage * kBoxBytes;
              return addr;
            };
            auto ring_done = [&]() {
              if (elect_one()) tc2::umma_commit(bar_b_empty + 8 * b_stage);
              if (++b_stage == kStages) { b_stage = 0; b_phase ^= 1; }
            };
            for (int kc = 0; kc < kchunks; ++kc) {
              a_wait(ct, kc);
              const uint32_t a3 = ring_wait();
              const uint32_t a3_stage = b_stage;
              uint32_t nxt = b_stage + 1 == kStages ? 0 : b_stage + 1;
              mbar_wait_batched(bar_b_full + 8 * nxt, nxt == 0 ? b_phase ^ 1 : b_phase);
              tc_fence_after();
              const uint32_t b1 = sbase + kSmemB + nxt * kBoxBytes;
              mma4(sbase + kSmemA + kc * kBoxBytes, b1);
              mma4(sbase + kSmemA + (kMaxKChunks + kc) * kBoxBytes, b1);
              mma4(a3, b1);
              (void)a3_stage;
              ring_done();                                         // a3[kc]
              ring_done();                                         // b1[kc]
            }
            for (int kc = 0; kc < kchunks; ++kc) {
              const uint32_t b2 = ring_wait();
              mma4(sbase + kSmemA + kc * kBoxBytes, b2);
              mma4(sbase + kSmemA + (kMaxKChunks + kc) * kBoxBytes, b2);
              ring_done();
            }
            for (int kc = 0; kc < kchunks; ++kc) {
              const uint32_t b3 = ring_wait();
              mma4(sbase + kSmemA + kc * kBoxBytes, b3);
              ring_done();
              a_done(ct, kc);                                      // (the a2 chunk was last read in the loop above)
            }
          } else
          for (int kc = 0; kc < kchunks; ++kc) {
            a_wait(ct, kc);
            mbar_wait_batched(bar_b_full + 8 * b_stage, b_phase);
            tc_fence_after();
            const uint32_t a_addr = sbase + kSmemA + kc * kBoxBytes;
            const uint32_t b_addr = sbase + kSmemB + b_stage * kBoxBytes;
            if (elect_one()) {
#pragma unroll
              for (int ks = 0; ks < kBoxK / 16; ++ks)
                tc2::umma_bf16(d, umma_desc(a_addr + ks * 32), umma_desc(b_addr + ks * 32), kIdesc, (kc | ks) ? 1u : 0u);
              tc2::umma_commit(bar_b_empty + 8 * b_stage);  // ring slot free in both CTAs once these MMAs have read it
            }
            a_done(ct, kc);
            if (++b_stage == kStages) { b_stage = 0; b_phase ^= 1; }
          }
          if (elect_one()) tc2::umma_commit(bar_acc_full + 8 * s);         // accumulator stage complete (both CTAs' epilogues)
        }
        a_phase ^= 1;
      }
    }
  } else if (warp == kWarpMma + 1) {
    // =============================== TMA loader of the stationary operand (both CTAs) ===============================
    // A thread of its own: the loads of a unit's block wait for MMAs that the streamed operand's producer is two tiles
    // ahead of, so they cannot share a queue with it.
    if (lane == 0) {
      uint32_t a_phase = 0;
      for (int u = pair; u < P.total_units; u += npairs) {
        int dir, n, rb;
        decode(u, dir, n, rb);
        if (skip_pair(n)) continue;
        const CUtensorMap* mapA = dir ? &map1 : &map0;
        const int arow = rb * kUnitRows + int(rank) * kBoxRows;
        for (int kc = 0; kc < kchunks; ++kc) {
          mbar_wait_batched(bar_a_empty + 8 * kc, a_phase ^ 1);
          if (rank == 0) mbar_expect_tx(bar_a_full + 8 * kc, (MODE == 4 ? 4 : 2) * kBoxBytes);
          tc2::tma_load_3d_2sm(sbase + kSmemA + kc * kBoxBytes, mapA, bar_a_full + 8 * kc, kc * kBoxK, arow, n);
          if (MODE == 4)      // a2 block behind the a1 block
            tc2::tma_load_3d_2sm(sbase + kSmemA + (kMaxKChunks + kc) * kBoxBytes, &map1, bar_a_full + 8 * kc, kc * kBoxK, arow, n);
        }
        a_phase ^= 1;
      }
    }
  }
  // (warp 19 only completes the last warpgroup)
  } else {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsEpi));
  if (MODE == 3 || MODE == 4) {
    // =============================== single-sweep epilogue (16 warps: 4 lane quadrants x 4 groups of 64 columns) =====
    // Every warp keeps one integer-valued shift m for its 32 rows: e = 2^(x - m).  Before the exponentials of a chunk each
    // thread takes the maximum of its 32 raw accumulators (16 three-input FMNMX); if any of them would land above 2^110 the
    // warp raises m to (chunk maximum - 96) and rescales its running row sums by that exact power of two -- so nothing ever
    // overflows and nothing is computed twice.  m is chosen from the data at the first chunk of a unit and never lowered.
    // Column sums leave the warp once per chunk together with the shift they were taken at; the merge kernel combines them.
    const int g = lane >> 2, p = lane & 3;
    const int cg = warp >> 2, quad = warp & 3;
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    float2* mergef = reinterpret_cast<float2*>(smem + kSmemMerge);   // [3][128] (row sum, shift) of column groups 1..3
    const int rin = quad * 32 + g + 8 * p;                           // the row of the CTA this lane writes results for
    // [128] per row of the CTA: log2 of the largest partial row sum any column group has published + kBndBias (float bits
    // compared as integers: positive floats order like their bits; 0 = nothing yet)
    constexpr float kBndBias = 16384.f;
    int* rowbnd = reinterpret_cast<int*>(smem + kSmemLc);
    const uint32_t rowbnd_addr = sbase + kSmemLc + 4 * (quad * 32 + g);   // this thread's rows: + 32 bytes per rho
    if (threadIdx.x < 128) rowbnd[threadIdx.x] = 0;
    asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
    const float scale = P.scale_log2, inv_scale = 1.f / P.scale_log2;
    const float thrm = exp2f(P.log2_thr) * 0.99f;
    const int LA = P.L0, LB = P.L1;
    const int ntiles = (LB + kTileCols - 1) / kTileCols, ngroups = (LA + 31) / 32, nblk = (LB + 31) / 32;
    const int ccol = 8 * (g >> 1) + 2 * p + (g & 1);                 // chunk column whose sum ss_col_reduce leaves in this lane
    // (made opaque: the compiler otherwise re-derives these from SR_TID.X for every tile -- ~40 instructions per tile --
    //  instead of spending two registers on them)
    uint32_t tb0 = tmem_base + lane_addr + cg * kSpan;               // TMEM address of the thread's columns in stage 0
    int colofs = cg * kSpan;                                         // the warp's first column within a tile
    asm volatile("" : "+r"(tb0), "+r"(colofs));
    uint32_t tile_ctr = 0;
    for (int u = pair; u < P.total_units; u += npairs) {
      int dir, n, rb;
      decode(u, dir, n, rb);
      const int rowbase = rb * kUnitRows + int(rank) * kBoxRows + quad * 32;
      const int rows_valid = min(max(LA - rowbase, 0), 32);
      uint32_t rowmask = 0;
#pragma unroll
      for (int rho = 0; rho < 4; ++rho) rowmask |= (g + 8 * rho < rows_valid) ? (1u << rho) : 0u;
      float rowacc[4] = {0.f, 0.f, 0.f, 0.f};                        // the thread's row sums (its 2 of every 8 columns)
      float tb[4] = {0.f, 0.f, 0.f, 0.f};                            // thr x (what is known of the rest of the row's sum)
      float mshift = 0.f, rawlim = -INFINITY;                        // raw accumulators above rawlim raise the shift (first chunk: always)
      uint32_t cnts = 0;                                             // fill counts of the thread's four private lists (a byte each)
      const uint32_t gidx = uint32_t(n) * ngroups + (rowbase >> 5);  // (pair, 32-row group): row of colpart / cshift
      // where this lane's column sum / this warp's shift of the current tile's first chunk go (advanced tile by tile)
      float* cp_ptr = P.colpart + size_t(gidx) * LB + (colofs + ccol);
      float* cs_ptr = P.cshift + size_t(gidx) * nblk + (colofs >> 5);
      // the thread's private candidate list of row (g + 8 rho) starts at listbase + rho * (8 rows of lists)
      u64* const listbase = P.cand + (((size_t(n) * LA + rowbase + g) * kListGroups + cg) * 4 + p) * kLaneSlots;

      for (int ct = 0; ct < ntiles; ++ct, ++tile_ctr) {
        const uint32_t s = tile_ctr & 1, acc_phase = (tile_ctr >> 1) & 1;
        const int col0 = ct * kTileCols;
        const int nvalid = min(LB - col0, kTileCols) - colofs;
        const bool active = rows_valid > 0 && nvalid > 0;
        mbar_wait_batched(bar_acc_full + 8 * s, acc_phase);
        tc_fence_after();
        const uint32_t tbase = tb0 + s * kTileCols;
        float v[32];
        auto process = [&](float (&v)[32], int cc) {
          const int vc = nvalid - cc * 32;
          const int colb = col0 + colofs + cc * 32;
          if (rows_valid < 32 || vc < 32) ss_mask(v, rowmask, vc, p);
          // ---- shift guard on the raw accumulators
          float t0 = fmax3(v[0], v[1], v[2]), t1 = fmax3(v[3], v[4], v[5]);
#pragma unroll
          for (int j = 6; j < 30; j += 4) {
            t0 = fmax3(t0, v[j], v[j + 1]);
            t1 = fmax3(t1, v[j + 2], v[j + 3]);
          }
          t0 = fmax3(t0, v[30], v[31]);
          const float tmax = fmaxf(t0, t1);
          if (__any_sync(kFullMask, tmax > rawlim)) {
            float cm = tmax;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) cm = fmaxf(cm, __shfl_xor_sync(kFullMask, cm, o));
            const bool first = rawlim == -INFINITY;                  // first chunk of the unit: no sums yet, any shift
            float mnew = floorf(cm * scale) - kShiftBack;
            if (!first) mnew = fmaxf(mnew, mshift);                  // afterwards the shift only rises
            if (!(fabsf(mnew) < 1e30f)) mnew = first ? 0.f : mshift; // inf inputs: the sums get flagged
            if (!first) {
#pragma unroll
              for (int rho = 0; rho < 4; ++rho) {
                rowacc[rho] = scale_pow2(rowacc[rho], mshift - mnew);
                tb[rho] = scale_pow2(tb[rho], mshift - mnew);
              }
            }
            mshift = mnew;
            rawlim = (mnew + kShiftHead) * inv_scale;
          }
          // ---- exponentials, row and column sums
          u64 cp2[4], rc2[4];
          ss_chunk(v, scale, -mshift, rc2, cp2);
          float cp[8];
#pragma unroll
          for (int k = 0; k < 4; ++k) unpack2(cp2[k], cp[2 * k], cp[2 * k + 1]);
          const float cs = ss_col_reduce(cp, lane);
          if (ccol < vc) cp_ptr[cc * 32] = cs;
          if (lane == 0) cs_ptr[cc] = mshift;
          // ---- candidates.  A cell can only have p_row > thr if it exceeds thr x (a lower bound of the row's final sum).
          // Level 1, no communication: this chunk's contribution d[rho] to the thread's own row sum against thr x (that sum
          // + what the thread last learnt about the rest of the row, tb[]); true for the first chunks of a unit by
          // construction.  Level 2, per row position rho and only if some lane passed level 1 for it: the row sum over the 4
          // lanes that share the row, and what the other column groups of the CTA have published about the row (rowbnd:
          // log2 of a partial row sum + kBndBias, raised with a shared-memory atomicMax; ANY lower bound of the final row
          // sum is a valid pruning bound, whenever it was taken).  Level 3: only a CELL above the bound is a candidate, so
          // the row's largest cell decides, and the lists are touched for real candidates only.  One cell above the bound
          // (the rest of the contribution cannot hold another one) is stored in line; several cells, or a full list, go
          // through the out-of-line scan.
          float d[4];
          bool pass = false;
#pragma unroll
          for (int rho = 0; rho < 4; ++rho) {
            float x, y;
            unpack2(rc2[rho], x, y);
            d[rho] = x + y;
            rowacc[rho] += d[rho];
            pass |= d[rho] > fmaf(thrm, rowacc[rho], tb[rho]);
          }
          if (__any_sync(kFullMask, pass)) {       // (one vote per chunk on the common path)
#pragma unroll
            for (int rho = 0; rho < 4; ++rho) {
              if (!__any_sync(kFullMask, d[rho] > fmaf(thrm, rowacc[rho], tb[rho]))) continue;
              float rs = rowacc[rho];
              rs += __shfl_xor_sync(kFullMask, rs, 1);
              rs += __shfl_xor_sync(kFullMask, rs, 2);
              const float other = ex2_approx(lds32(rowbnd_addr + 32 * rho) - (kBndBias + mshift));
              const float bound = thrm * fmaxf(rs, other);
              tb[rho] = fmaxf(tb[rho], fmaf(-thrm, rowacc[rho], bound));
              if (p == 0 && fabsf(mshift) < 0.5f * kBndBias)     // (explicit shared-space reduction: through the
                red_max_shared(rowbnd_addr + 32 * rho,          //  generic pointer it compiled to ATOM.E...GPU)
                               __float_as_int(lg2_approx(rs) + (mshift + kBndBias - 0.004f)));
              const int i0 = 16 * (rho >> 1) + 2 * (rho & 1);
              const float e0 = v[i0], e1 = v[i0 + 1], e2 = v[i0 + 4], e3 = v[i0 + 5], e4 = v[i0 + 8], e5 = v[i0 + 9],
                          e6 = v[i0 + 12], e7 = v[i0 + 13];
              const float emax = fmax3(fmax3(e0, e1, e2), fmax3(e3, e4, e5), fmaxf(e6, e7));
              if (emax > bound) {
                u64* const mylist = listbase + rho * (8 * kListGroups * 4 * kLaneSlots);
                int c = int((cnts >> (8 * rho)) & 0xffu);
                if (d[rho] - emax <= bound && c < kLaneSlots) {
                  int q = 0;
                  q = e1 == emax ? 1 : q; q = e2 == emax ? 2 : q; q = e3 == emax ? 3 : q; q = e4 == emax ? 4 : q;
                  q = e5 == emax ? 5 : q; q = e6 == emax ? 6 : q; q = e7 == emax ? 7 : q;
                  const int col = colb + 2 * p + 8 * (q >> 1) + (q & 1);
                  mylist[c] = (u64(__float_as_uint(log2_split(emax) + mshift)) << 32) | uint32_t(col);
                  ++c;
                } else {
                  c = ss_scan_row(e0, e1, e2, e3, e4, e5, e6, e7, bound, mshift, mylist, c, colb + 2 * p, P.flags, P.pairflag + n);
                }
                cnts = (cnts & ~(0xffu << (8 * rho))) | (uint32_t(c) << (8 * rho));
              }
            }
          }
        };
        if (active) {
          tmem_ld_frag(tbase, v);
          process(v, 0);
        }
        if (active && nvalid > 32) tmem_ld_frag(tbase + 32, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) tc2::mbar_arrive_leader(bar_acc_empty + 8 * s);
        if (active && nvalid > 32) process(v, 1);
        cp_ptr += kTileCols;
        cs_ptr += kTileCols / 32;
      }

      // unit end: row sums over the 4 lanes of a row (same warp, same shift), then over the 4 column groups (one shift
      // each) through shared memory
#pragma unroll
      for (int rho = 0; rho < 4; ++rho) {
        rowacc[rho] += __shfl_xor_sync(kFullMask, rowacc[rho], 1);
        rowacc[rho] += __shfl_xor_sync(kFullMask, rowacc[rho], 2);
      }
      const float mine = p == 0 ? rowacc[0] : p == 1 ? rowacc[1] : p == 2 ? rowacc[2] : rowacc[3];
      // list counts: row (g + 8 rho)'s uint16 = the nibbles of its four lanes; lane p publishes row rho = p
      uint32_t myfield = 0;
#pragma unroll
      for (int rho = 0; rho < 4; ++rho) {
        uint32_t f = ((cnts >> (8 * rho)) & 0xfu) << (4 * p);
        f |= __shfl_xor_sync(kFullMask, f, 1);
        f |= __shfl_xor_sync(kFullMask, f, 2);
        myfield = (p == rho) ? f : myfield;
      }
      if (cg > 0) mergef[(cg - 1) * 128 + rin] = make_float2(mine, mshift);
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      const int row = rb * kUnitRows + int(rank) * kBoxRows + rin;
      if (row < LA) {
        if (cg == 0) {
          // domain of the total = the largest shift among the column groups that hold anything
          float sk[4] = {mine, 0.f, 0.f, 0.f}, mk[4] = {mshift, 0.f, 0.f, 0.f};
#pragma unroll
          for (int q = 1; q < 4; ++q) {
            const float2 t = mergef[(q - 1) * 128 + rin];
            sk[q] = t.x;
            mk[q] = t.y;
          }
          float mtop = -INFINITY;
#pragma unroll
          for (int q = 0; q < 4; ++q) mtop = (sk[q] != 0.f) ? fmaxf(mtop, mk[q]) : mtop;
          float tot = 0.f;
#pragma unroll
          for (int q = 0; q < 4; ++q) tot += (sk[q] != 0.f) ? scale_pow2(sk[q], mk[q] - mtop) : 0.f;
          P.lse_out0[size_t(n) * LA + row] = mtop + log2f(tot);
          if (!(tot > kSumLo && tot < kSumHi)) {
            atomicOr(reinterpret_cast<unsigned*>(P.flags), POPE_FLAG_ROBUST_PATH);
            *reinterpret_cast<volatile int*>(P.pairflag + n) = 1;
          }
        }
        reinterpret_cast<uint16_t*>(P.cand_cnt)[(size_t(n) * LA + row) * kListGroups + cg] = uint16_t(myfield);
      }
      if (threadIdx.x < 128) rowbnd[threadIdx.x] = 0;                 // (every warp is past its last tile of the unit)
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
    }
  } else {
    // =============================== epilogue (16 warps; four threads per row, 64 columns of the tile each) =========
    constexpr bool kLse = (MODE == 0 || MODE == 2);      // online log-sum-exp of the thread's row
    constexpr bool kStage = (MODE == 1);                 // per-column terms staged in shared memory (three-sweep path)
    const int e = threadIdx.x;                      // 0..511
    const int colq = warp >> 2;                     // which kSpan of the tile's 256 columns (4 consecutive warps = 4 quadrants)
    const int quad = warp & 3;                      // TMEM lane quadrant this warp may touch
    const int row_in_cta = quad * 32 + lane;
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    float* lc_bound = reinterpret_cast<float*>(smem + kSmemLc);          // [2][256] pre-filter bounds
    float* lc_exact = lc_bound + 2 * kTileCols;                          // [2][256] exact column log-sum-exp (MODE 1)
    float2* merge = reinterpret_cast<float2*>(smem + kSmemMerge);        // [3][128] (max, sum) of column quarters 1..3
    uint32_t tile_ctr = 0;
    for (int u = pair; u < P.total_units; u += npairs) {
      int dir, n, rb;
      decode(u, dir, n, rb);
      if (skip_pair(n)) continue;
      const int LA = dir ? P.L1 : P.L0, LB = dir ? P.L0 : P.L1;
      const int ntiles = (LB + kTileCols - 1) / kTileCols;
      const int row = rb * kUnitRows + int(rank) * kBoxRows + row_in_cta;
      const float scale = P.scale_log2;
      const float* col_term = P.lse_c;      // MODE 1: per-column term lse_c, this thread's row term lse_r added per thread
      const float inv_s = 1.f / (2.f * scale);
      const bool listing = (MODE == 2) && dir == 0 && row < LA;     // MODE 2: this thread lists candidates of its row
      const float inv_scale = 1.f / scale;
      u64* const mylist = P.cand + ((size_t(n) * LA + row) * kListGroups + colq) * kListStride;
      int list_cnt = 0;

      float m_run = -INFINITY, s_run = 0.f;         // log-sum-exp state
      float lrp = INFINITY, lr = INFINITY;
      float lc_next = INFINITY;
      if (kStage) {
        if (MODE == 1 && row < LA) {
          lr = P.lse_r[size_t(n) * LA + row];
          const float b = (lr + P.log2_thr) * inv_s;
          lrp = isfinite(b) ? b - 1e-5f * fabsf(b) - 0.005f * inv_s : INFINITY;
        }
        if (e < kTileCols && e < LB) lc_next = __ldg(col_term + size_t(n) * LB + e);
      }

      for (int ct = 0; ct < ntiles; ++ct, ++tile_ctr) {
        const uint32_t s = tile_ctr & 1, acc_phase = (tile_ctr >> 1) & 1;
        const int col0 = ct * kTileCols;
        if (kStage) {
          // stage this tile's column terms (fetched one tile ahead) as pre-filter bounds in raw-accumulator units,
          // margin on the safe side, +inf past the last column
          if (e < kTileCols) {
            const float b = lc_next * inv_s;
            lc_exact[s * kTileCols + e] = lc_next;
            lc_bound[s * kTileCols + e] = isfinite(b) ? b - 1e-5f * fabsf(b) : INFINITY;
            const int coln = col0 + kTileCols + e;
            lc_next = (coln < LB) ? __ldg(col_term + size_t(n) * LB + coln) : INFINITY;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        }
        mbar_wait_batched(bar_acc_full + 8 * s, acc_phase);
        tc_fence_after();
        const uint32_t tbase = tmem_base + lane_addr + s * kTileCols + colq * kSpan;
        const int nvalid = min(LB - col0, kTileCols) - colq * kSpan;   // valid columns from this thread's first one
        if (MODE == 1) {
          // ---- three-sweep path: candidate test against both log-sum-exps; flagged columns re-read from TMEM ----
#pragma unroll 1
          for (int cc = 0; cc < kChunks; ++cc) {
            const int vc = nvalid - cc * 32;
            if (vc <= 0) break;
            float v[32];
            tmem_ld32(tbase + cc * 32, v);
            const uint32_t lb = sbase + kSmemLc + (s * kTileCols + colq * kSpan + cc * 32) * 4;
            bool any = false;
#pragma unroll
            for (int j4 = 0; j4 < 32; j4 += 4) {
              const float4 l4 = lds128(lb + j4 * 4);
              any |= (v[j4 + 0] > lrp + l4.x) | (v[j4 + 1] > lrp + l4.y) | (v[j4 + 2] > lrp + l4.z) | (v[j4 + 3] > lrp + l4.w);
            }
            if (__any_sync(kFullMask, any)) {
              uint32_t mask = 0;
#pragma unroll
              for (int j = 0; j < 32; ++j) mask |= (v[j] > lrp + lds32(lb + j * 4)) ? (1u << j) : 0u;
              uint32_t all = __reduce_or_sync(kFullMask, mask);
              while (all) {
                const int j = __ffs(all) - 1;
                all &= all - 1;
                const float vj = tmem_ld1(tbase + cc * 32 + j);
                if ((mask >> j) & 1u) {
                  const int col = col0 + colq * kSpan + cc * 32 + j;
                  const float x = vj * scale;
                  const float t2 = (x - lr) + (x - lc_exact[s * kTileCols + colq * kSpan + cc * 32 + j]);
                  if (t2 > P.log2_thr) {
                    atomicMax(P.rowbest + size_t(n) * LA + row, pack_best(t2, col));
                    atomicMax(P.colbest + size_t(n) * LB + col, pack_best(t2, row));
                  }
                }
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) tc2::mbar_arrive_leader(bar_acc_empty + 8 * s);
        } else {
          // ---- log-sum-exp sweeps: the accumulator stage is handed back to the MMA issuer as soon as this warp's
          //      last TMEM load has retired; the second chunk's arithmetic and every atomic run after the hand-back ----
          auto scan = [&](const float (&v)[32], int cc, int vc, float cmax) {
            // MODE 2: cells above thr x (running row sum, this chunk included).  One MUFU.LG2 + a compare per chunk; the
            // per-element scan runs only for the threads whose chunk maximum passes (the row's match, typically once).
            const float b = (m_run + lg2_approx(s_run) + P.log2_thr) * inv_scale;
            const float bound = isfinite(b) ? b - (1e-5f * fabsf(b) + 0.005f * inv_scale) : INFINITY;
            if (cmax > bound) {
              const int colb = col0 + colq * kSpan + cc * 32;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (v[j] > bound && j < vc)
                  list_cnt = list_push<kCandSlots>(mylist, list_cnt, bound * scale, v[j] * scale, colb + j, P.flags, nullptr);
            }
          };
          static_assert(kChunks == 2, "the chunk-by-chunk epilogue is written for two chunks per thread");
          const int vc0 = nvalid, vc1 = nvalid - 32;
          float v[32];
          if (vc0 > 0) {
            tmem_ld32(tbase, v);
            const float cmax = lse_update(v, vc0, scale, m_run, s_run);
            if (listing) scan(v, 0, vc0, cmax);
          }
          if (vc1 > 0) tmem_ld32(tbase + 32, v);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) tc2::mbar_arrive_leader(bar_acc_empty + 8 * s);
          if (vc1 > 0) {
            const float cmax = lse_update(v, vc1, scale, m_run, s_run);
            if (listing) scan(v, 1, vc1, cmax);
          }
        }
      }
      if (listing)      // nibble counts of the quarter's sub-lists: the thread's entries are contiguous from entry 0
        reinterpret_cast<uint16_t*>(P.cand_cnt)[(size_t(n) * LA + row) * kListGroups + colq] =
            uint16_t(min(list_cnt, kLaneSlots) | (max(list_cnt - kLaneSlots, 0) << 4));
      if (kLse) {
        // the four column quarters of a row merge their (max, sum) through shared memory
        if (colq > 0) merge[(colq - 1) * 128 + row_in_cta] = make_float2(m_run, s_run);
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        if (colq == 0 && row < LA) {
          float m = m_run, sum = s_run;
#pragma unroll
          for (int q = 0; q < kColGroups - 1; ++q) {
            const float2 o = merge[q * 128 + row_in_cta];
            const float mm = fmaxf(m, o.x);
            sum = sum * ex2_approx(m - mm) + o.y * ex2_approx(o.x - mm);
            m = mm;
          }
          (dir ? P.lse_out1 : P.lse_out0)[size_t(n) * LA + row] = m + lg2_approx(sum);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      }
    }
  }

  }

  tc_fence_before();
  __syncthreads();
  tc2::cluster_sync_all();                           // the peer may still be signalling / reading this CTA's memory
  if (warp == kWarpMma) {
    tc_fence_after();
    tc2::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// fp32 -> three bf16 planes with a = a1 + a2 + a3 (each residual is exact in fp32): 8 + 8 + 8 mantissa bits
__global__ void __launch_bounds__(256) split3_kernel(const float4* __restrict__ in, uint2* __restrict__ p1, uint2* __restrict__ p2,
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

// ---- host side ------------------------------------------------------------------------------------------------------
// [n, rows, C] bf16, box = 64 k x 128 rows x 1 pair, 128-byte swizzle, zero fill past the last row
bool make_map(CUtensorMap* m, const void* base, int n, int rows, int C) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return false;
  cuuint64_t dims[3] = {cuuint64_t(C), cuuint64_t(rows), cuuint64_t(n)};
  cuuint64_t strides[2] = {cuuint64_t(C) * 2, cuuint64_t(rows) * C * 2};
  cuuint32_t box[3] = {kBoxK, kBoxRows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Test hooks (environment variable POPE_TC_DEBUG), the references the tests hold the product sequence to:
//   16   = no single sweep: the two-sweep online-softmax launch runs ungated, for every pair (bf16 features);
//   1024 = the single sweep runs as one launch, without the head / tail cut (bf16 and fp32 features).
constexpr int kHookTwoSweeps = 16, kHookOneLaunch = 1024;
int debug_knob() {
  const char* dbg = getenv("POPE_TC_DEBUG");
  return dbg ? atoi(dbg) : 0;
}

// Head/tail cut of the single sweep (see single_sweep_run): the number of leading pairs whose units fill whole rounds of the
// static schedule, or 0 when the sweep should stay one launch.
int split_head(int n, int upp, int max_pairs) {
  const int u0 = n * upp;
  if (n <= 1 || u0 <= max_pairs || u0 % max_pairs == 0) return 0;
  const int rounds = (u0 + max_pairs - 1) / max_pairs;
  const int h = ((u0 / max_pairs) * max_pairs) / upp;                          // pairs that fit the full rounds
  const int ua = h * upp, ub = u0 - ua;
  if (h > 0 && h < n && (ua + max_pairs - 1) / max_pairs + (ub + max_pairs - 1) / max_pairs == rounds &&
      2 * ub <= max_pairs + max_pairs / 2)
    return h;
  return 0;
}

using SweepKernel = decltype(&sweep_tc_kernel<0>);

// per-device attribute, cheap: set on every call so that any device of a multi-GPU process is covered
cudaError_t allow_smem(SweepKernel k) { return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemAlloc); }

// CTA pairs of the persistent sweeps on the current device: one per two SMs
cudaError_t cta_pairs(int* max_pairs) {
  int dev = 0, sms = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  *max_pairs = sms / 2;
  return cudaSuccess;
}

// the parameters every sweep launch shares; the pairs, units and gate are set per launch
SweepParams sweep_params(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags) {
  SweepParams P{};
  P.n = p.n; P.L0 = p.L; P.L1 = p.S; P.kchunks = p.C / kBoxK;
  P.scale_log2 = p.scale_log2; P.log2_thr = p.log2_thr;
  P.lse_out0 = w.lse_r; P.lse_out1 = w.lse_c; P.lse_r = w.lse_r; P.lse_c = w.lse_c; P.rowbest = w.rowbest; P.colbest = w.colbest;
  P.cand_cnt = w.cand_cnt; P.cand = w.cand; P.flags = flags; P.colpart = w.colpart; P.cshift = w.cshift; P.pairflag = w.pairflag;
  return P;
}

// Single sweep over the rows of S (`kernel`: MODE 3 for bf16 features, MODE 4 for fp32 features as three bf16 planes) and
// the merge of its column partial sums into the column log-sum-exp.  Clears the pair flags; the merge resets colbest and
// the "count published" words itself, so rowbest..ready need no memset.  Raises POPE_FLAG_ROBUST_PATH when the exponentials
// of a pair leave the safe range.  The candidate lists are evaluated by the caller, behind the fallback of its dtype.
// The unit schedule is static: u0 units over max_pairs CTA pairs run in ceil(u0 / max_pairs) rounds, and the last round
// is usually part empty (64 pairs at 480x640: 1 216 units = 16 rounds of 74 + 32).  When the pairs can be cut into a
// head that fills whole rounds and a tail that fits the last round without adding one, the sweep is launched twice --
// head, then tail -- and the column merge of the head's pairs runs on the SMs the tail leaves idle: the sweep kernel
// announces its dependents at once (griddepcontrol.launch_dependents) and merge(head), which needs nothing from the
// tail (the head sweep has completed before the tail started), is launched behind the tail with programmatic stream
// serialisation: ONE merge launch over all pairs, whose blocks for the head's pairs never wait and whose blocks for the
// tail's pairs (the last of the grid) wait for the tail sweep (griddepcontrol.wait).  Everything behind it is ordinary.
cudaError_t single_sweep_run(SweepKernel kernel, const CUtensorMap (&m)[6], const CoarseProblem& p, const CoarseScratch& w,
                             int32_t* flags, cudaStream_t st) {
  int max_pairs = 0;
  cudaError_t e;
  if ((e = cta_pairs(&max_pairs)) != cudaSuccess) return e;
  if ((e = allow_smem(kernel)) != cudaSuccess) return e;
  const SweepParams P = sweep_params(p, w, flags);
  const int upp = (p.L + kUnitRows - 1) / kUnitRows;                           // units per pair
  if ((e = cudaMemsetAsync(w.pairflag, 0, sizeof(int) * p.n, st)) != cudaSuccess) return e;
  const int head = (debug_knob() & kHookOneLaunch) ? 0 : split_head(p.n, upp, max_pairs);
  auto sweep = [&](int n_base, int n_count) -> cudaError_t {
    SweepParams Q = P;
    Q.n_base = n_base; Q.n = n_count;
    Q.units_dir0 = Q.total_units = n_count * upp;
    kernel<<<2 * min(Q.total_units, max_pairs), kThreads, kSmemAlloc, st>>>(m[0], m[1], m[2], m[3], m[4], m[5], Q);
    return cudaGetLastError();
  };
  if (head > 0) {
    if ((e = sweep(0, head)) != cudaSuccess) return e;
    if ((e = sweep(head, p.n - head)) != cudaSuccess) return e;
    return colsum_reduce_run(p, w, flags, st, 0, p.n, head);
  }
  if ((e = sweep(0, p.n)) != cudaSuccess) return e;
  return colsum_reduce_run(p, w, flags, st, 0, p.n);
}
}  // namespace

bool coarse_tc_supported(const CoarseProblem& p) {
  return p.dtype == POPE_BF16 && p.C % kBoxK == 0 && p.C >= kBoxK && p.C <= kBoxK * kMaxKChunks;
}

// fp32 features on the tensor cores through the three-way bf16 split (single-sweep path only: thr > 0.15)
bool coarse_tc_split_supported(const CoarseProblem& p) {
  return p.dtype == POPE_F32 && p.C % kBoxK == 0 && p.C >= kBoxK && p.C <= kBoxK * kMaxKChunks && two_sweeps_possible(p);
}

size_t coarse_tc_split_bytes(int n, int L, int S, int C) { return 3 * 2 * (size_t(n) * L * C + size_t(n) * S * C) + 6 * 256; }

// planes: 3 x [n, L, C] then 3 x [n, S, C] bf16 in `planes` (coarse_tc_split_bytes).  Single sweep; if the sums leave the safe
// range the flag is raised and the caller's gated fp32-FMA launches redo the batch.
cudaError_t coarse_tc_split_run(const CoarseProblem& p, const CoarseScratch& w, void* planes, int32_t* flags, cudaStream_t st) {
  const size_t e0 = size_t(p.n) * p.L * p.C, e1 = size_t(p.n) * p.S * p.C;
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  char* base = static_cast<char*>(planes);
  __nv_bfloat16* pl[6];
  size_t off = 0;
  for (int k = 0; k < 6; ++k) { pl[k] = reinterpret_cast<__nv_bfloat16*>(base + off); off += up((k < 3 ? e0 : e1) * 2); }
  cudaError_t e;
  split3_kernel<<<148 * 8, 256, 0, st>>>(static_cast<const float4*>(p.f0), reinterpret_cast<uint2*>(pl[0]),
                                         reinterpret_cast<uint2*>(pl[1]), reinterpret_cast<uint2*>(pl[2]), e0 / 4);
  split3_kernel<<<148 * 8, 256, 0, st>>>(static_cast<const float4*>(p.f1), reinterpret_cast<uint2*>(pl[3]),
                                         reinterpret_cast<uint2*>(pl[4]), reinterpret_cast<uint2*>(pl[5]), e1 / 4);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  CUtensorMap m[6];
  for (int k = 0; k < 6; ++k)
    if (!make_map(&m[k], pl[k], p.n, k < 3 ? p.L : p.S, p.C)) return cudaErrorInvalidValue;
  if ((e = single_sweep_run(sweep_tc_kernel<4>, m, p, w, flags, st)) != cudaSuccess) return e;
  return cand_eval_lists_run(p, w, flags, 2, st);       // mode 2: 2^x lists; a no-op once the fallback flag is up
}

cudaError_t coarse_tc_run(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st) {
  CUtensorMap m[6];                                     // MODES 0-3 read the first two maps only
  if (!make_map(&m[0], p.f0, p.n, p.L, p.C) || !make_map(&m[1], p.f1, p.n, p.S, p.C)) return cudaErrorInvalidValue;
  m[2] = m[4] = m[0];
  m[3] = m[5] = m[1];
  int max_pairs = 0;
  cudaError_t e;
  if ((e = cta_pairs(&max_pairs)) != cudaSuccess) return e;
  SweepParams P = sweep_params(p, w, flags);
  const int u0 = p.n * ((p.L + kUnitRows - 1) / kUnitRows), u1 = p.n * ((p.S + kUnitRows - 1) / kUnitRows);
  auto launch = [&](SweepKernel k, int total_units) -> cudaError_t {
    if ((e = allow_smem(k)) != cudaSuccess) return e;
    P.units_dir0 = u0; P.total_units = total_units;
    k<<<2 * min(total_units, max_pairs), kThreads, kSmemAlloc, st>>>(m[0], m[1], m[2], m[3], m[4], m[5], P);
    return cudaGetLastError();
  };
  // A cell with conf > thr has p_row > thr, and a row has fewer than 1/thr such cells: with thr > 1/kCandSlots the
  // column sweep can list them and the third (candidate) sweep is not needed.
  if (two_sweeps_possible(p)) {
    if (debug_knob() & kHookTwoSweeps) {
      // without the single sweep's column merge nothing resets colbest and the "count published" words
      if ((e = cudaMemsetAsync(w.rowbest, 0, w.zero_bytes, st)) != cudaSuccess) return e;
    } else {
      // single sweep over the rows of S: row sums, column partial sums and candidate lists in one pass
      if ((e = single_sweep_run(sweep_tc_kernel<3>, m, p, w, flags, st)) != cudaSuccess) return e;
      P.gate = 1;
    }
    // robust two-sweep path (online softmax per row, both directions in one launch; the direction-0 units also fill the
    // per-thread candidate lists); after the single sweep it only runs if the flag was raised
    if ((e = launch(sweep_tc_kernel<2>, u0 + u1)) != cudaSuccess) return e;
    return cand_eval_lists_run(p, w, flags, 0, st);
  }
  // three sweeps (small thresholds): both log-sum-exp directions in one launch, then the candidate sweep
  if ((e = cudaMemsetAsync(w.rowbest, 0, w.zero_bytes, st)) != cudaSuccess) return e;
  if ((e = launch(sweep_tc_kernel<0>, u0 + u1)) != cudaSuccess) return e;
  return launch(sweep_tc_kernel<1>, u0);
}

}  // namespace pope
