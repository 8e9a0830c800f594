// common.cuh -- shared device helpers and internal launcher declarations of libpope_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "pope_b200.h"

namespace pope {

typedef unsigned long long u64;

constexpr float kLog2e = 1.4426950408889634f;
constexpr unsigned kFullMask = 0xffffffffu;

// ---- order-preserving float <-> uint key (so that atomicMax on integers is a float max) -------------------
__device__ __forceinline__ uint32_t ordered_key(float t) {
  uint32_t b = __float_as_uint(t);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// Best-candidate record: high word = ordered log2-confidence, low word = ~index, so that atomicMax keeps the
// largest confidence and, on exact ties, the smallest index.  0 means "no candidate".
__device__ __forceinline__ u64 pack_best(float t2, int idx) {
  return (static_cast<u64>(ordered_key(t2)) << 32) | static_cast<uint32_t>(~static_cast<uint32_t>(idx));
}
__device__ __forceinline__ int best_index(u64 rec) { return static_cast<int>(~static_cast<uint32_t>(rec)); }
__device__ __forceinline__ uint32_t best_key(u64 rec) { return static_cast<uint32_t>(rec >> 32); }

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// x * 2^d for x >= 0 and an integer-valued d <= 0, by exponent arithmetic: exact, and correct when 2^d itself is below the
// normal range (a factor 2^-146 would flush to zero although 2^68 * 2^-146 is an ordinary number).  Results below 2^-126
// flush to zero; 0, inf and nan pass through.  Used wherever a sum moves to a higher shift domain.
__device__ __forceinline__ float scale_pow2(float x, float d) {
  const int b = __float_as_int(x);
  if (!(x > 0.f) || b >= 0x7f800000) return x;
  if (!(d > -280.f)) return 0.f;
  const int e = b + (int(d) << 23);
  return e >= 0x00800000 ? __int_as_float(e) : 0.f;
}

// ---- coarse-match scratch layout -------------------------------------------------------------------------
constexpr int kCandSlots = 8;   // per-row candidate slots of the two-sweep paths (thr > 1/8 => at most 7 cells pass)
// tcgen05 paths: every epilogue thread keeps PRIVATE candidate lists, so the sweeps need no atomics.  A row owns
// kListGroups (column quarters) x kListStride entries.  Two-sweep kernels: thread (row, quarter) fills the first kCandSlots
// entries of its quarter.  Single sweep: the four lanes that share a row in a quarter own kLaneSlots entries each -- at most
// 1 / (0.99 thr) cells of a row can exceed thr x (row sum) at any time (5 for thr = 0.2), and a full list is re-filtered
// against the current sum before it takes another cell, so six slots cannot overflow for thr > 1/6, wherever the cells fall.
// Counts: one uint16 per (row, quarter) = four nibbles, nibble p = entries used in sub-list p (entries [6p, 6p + 6)).
constexpr int kListGroups = 4;
constexpr int kListStride = 24;
constexpr int kLaneSlots = 6;
// single-sweep path: every epilogue warp keeps an integer-valued shift m (e = 2^(x - m)).  A fresh shift leaves the chunk's
// largest cell at 2^96, and no cell is ever allowed above 2^110 (the warp raises m first), so sums of <= 2^16 terms stay
// below 2^126.  The window is deliberately lopsided: the risk is at the bottom, where rows / columns whose maxima lie far
// below the strongest cell of their 32-row group underflow.  A term that underflows is below 2^-126 in its sum's final
// domain, so a row / column sum above 2^-90 of that domain has lost less than 2^-20 of its value; below it the pair is
// handed to the online-softmax kernels (POPE_FLAG_ROBUST_PATH): rows whose maxima are more than ~186 log2 units (129 in
// natural-log similarity) below the strongest row of their group.
constexpr float kSumLo = 8.0779357e-28f, kSumHi = 1.7014118e38f;
constexpr float kShiftBack = 96.f;           // a freshly chosen shift leaves the chunk's largest cell at 2^96
constexpr float kShiftHead = 110.f;          // a cell that would land above 2^110 raises the warp's shift first

struct CoarseScratch {
  float* lse_r;   // [n, L]  log2-domain log-sum-exp of every row of S
  float* lse_c;   // [n, S]  ... of every column
  u64* rowbest;   // [n, L]  best above-threshold candidate of the row   (pack_best(t2, j))
  u64* colbest;   // [n, S]  best above-threshold candidate of the column (pack_best(t2, i))
  int* cand_cnt;  // [n, L, 2]  tcgen05: four uint16 per row (above); SIMT: [n, L] ints, number of listed cells of the row
  u64* cand;      // [n, L, kListGroups, kListStride]  (tcgen05: similarity in log2 units, float bits << 32 | column); SIMT uses [n, L, kCandSlots] raw accumulators
  float* cbound;  // [n, 32*ceil(L/32)]  two-sweep path: raw-accumulator bound above which a cell of row i has p_row > thr
  float* cminb;   // [n, ceil(L/32)]  minimum of cbound over each group of 32 rows
  float* colpart; // [n, ceil(L/32), S]  single-sweep tcgen05 path: column sums of 2^(x - shift) over each group of 32 rows
  float* cshift;  // [n, ceil(L/32), ceil(S/32)]  ... the shift of each (32-row group, 32-column block) of colpart
  int* ready;     // [n + 1]  count_emit_kernel: "this pair's count is published", then its ticket counter (cleared before every call)
  int* pairflag;  // [n]  single-sweep path: != 0 = this pair is recomputed by the gated online-softmax launch
  size_t zero_bytes;   // rowbest, colbest, cand_cnt, ready are adjacent and cleared by one memset
  size_t bytes;
};
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline CoarseScratch carve_coarse_scratch(void* base, int n, int L, int S) {
  CoarseScratch w;
  char* p = static_cast<char*>(base);
  size_t off = 0;
  w.rowbest = reinterpret_cast<u64*>(p + off); off += align_up(sizeof(u64) * size_t(n) * L, 256);
  w.colbest = reinterpret_cast<u64*>(p + off); off += align_up(sizeof(u64) * size_t(n) * S, 256);
  w.cand_cnt = reinterpret_cast<int*>(p + off); off += align_up(sizeof(int) * size_t(n) * L * 2, 256);
  w.ready = reinterpret_cast<int*>(p + off); off += align_up(sizeof(int) * (size_t(n) + 1), 256);
  w.zero_bytes = off;
  w.lse_r = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * L, 256);
  w.lse_c = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * S, 256);
  w.cand = reinterpret_cast<u64*>(p + off); off += align_up(sizeof(u64) * size_t(n) * L * kListGroups * kListStride, 256);
  w.cbound = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * ((L + 31) / 32) * 32, 256);
  w.cminb = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * ((L + 31) / 32), 256);
  w.colpart = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * ((L + 31) / 32) * S, 256);
  w.cshift = reinterpret_cast<float*>(p + off); off += align_up(sizeof(float) * size_t(n) * ((L + 31) / 32) * ((S + 31) / 32), 256);
  w.pairflag = reinterpret_cast<int*>(p + off); off += align_up(sizeof(int) * size_t(n), 256);
  w.bytes = off;
  return w;
}

struct CoarseProblem {
  const void* f0;  // [n, L, C]
  const void* f1;  // [n, S, C]
  int dtype, n, L, S, C;
  int h0c, w0c, h1c, w1c;
  float scale_log2;  // log2(e) / (C * temperature): S in log2 units = <f0,f1> * scale_log2
  float log2_thr;    // log2(float(thr))
  int border;
  float pixel_scale;
};

// coarse_simt.cu -- fp32-FMA kernels (fp32 or bf16 inputs): the fp32 product path and the cross-check for tcgen05.
// gated: every launch is a no-op unless POPE_FLAG_ROBUST_PATH is set in *flags (the fallback of the fp32 tensor-core path).
// Both forms start by clearing the best-candidate records and counters themselves (the gated one only behind the flag).
cudaError_t coarse_simt_run(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st, bool gated = false);
// coarse_tc.cu -- tcgen05/TMEM/TMA kernels (bf16 inputs, C in {64,128,192,256})
bool coarse_tc_supported(const CoarseProblem& p);
// fp32 features through the three-way bf16 split (fp32 accuracy on the bf16 tensor cores); planes: extra scratch
bool coarse_tc_split_supported(const CoarseProblem& p);
size_t coarse_tc_split_bytes(int n, int L, int S, int C);
cudaError_t coarse_tc_split_run(const CoarseProblem& p, const CoarseScratch& w, void* planes, int32_t* flags, cudaStream_t st);
cudaError_t coarse_tc_run(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st);
// coarse_finalize.cu -- two-sweep helpers (shared by both kernel families): per-row bounds for the column sweep's
// candidate test, and the evaluation of the listed candidates
cudaError_t cand_bounds_run(const CoarseProblem& p, const CoarseScratch& w, cudaStream_t st, const int32_t* gate = nullptr);
cudaError_t cand_eval_run(const CoarseProblem& p, const CoarseScratch& w, cudaStream_t st, const int32_t* gate = nullptr);
// zero `bytes` (multiple of 16) at ptr if POPE_FLAG_ROBUST_PATH is set in *gate
cudaError_t gated_clear_run(void* ptr, size_t bytes, const int32_t* gate, cudaStream_t st);
// evaluation of the per-thread (row, column quarter) lists written by the tcgen05 row sweep
// (the lists hold raw accumulators on every path; mode 2 = fp32 split path: nothing at all if POPE_FLAG_ROBUST_PATH is set,
//  the fp32-FMA fallback evaluates its own lists)
cudaError_t cand_eval_lists_run(const CoarseProblem& p, const CoarseScratch& w, const int32_t* flags, int mode, cudaStream_t st);
// single-sweep tcgen05 path: column log-sum-exp from the per-32-row partial sums and their shifts (a log-sum-exp merge);
// sets POPE_FLAG_ROBUST_PATH and the pair's flag when a column sum lost precision
// (pairs [n_base, n_base + n_count) only: the single sweep may be launched in two parts)
// wait_from >= 0: launched with programmatic stream serialisation, i.e. the kernel may start while the kernel in front of it
// (the tail of a split single sweep) still runs; only the blocks of the pairs >= wait_from wait for that kernel
cudaError_t colsum_reduce_run(const CoarseProblem& p, const CoarseScratch& w, int32_t* flags, cudaStream_t st, int n_base, int n_count,
                              int wait_from = -1);
// a thr large enough that a row's cells with p_row > thr fit its kCandSlots candidate slots
inline bool two_sweeps_possible(const CoarseProblem& p) { return exp2f(p.log2_thr) * float(kCandSlots) > 1.2f; }
// coarse_finalize.cu -- mutual test, border removal, ordered compaction
cudaError_t coarse_finalize_run(const CoarseProblem& p, const CoarseScratch& w, int64_t* b_ids, int64_t* i_ids,
                                int64_t* j_ids, float* mconf, float* mk0, float* mk1, int32_t* counts, int64_t capacity,
                                cudaStream_t st);

}  // namespace pope
