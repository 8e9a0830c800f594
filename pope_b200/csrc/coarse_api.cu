// coarse_api.cu -- C-ABI entry points for coarse matching (argument checking, scratch carving, dispatch).
#include <math.h>

#include "common.cuh"

using namespace pope;

extern "C" int pope_abi_version(void) { return POPE_B200_ABI_VERSION; }

extern "C" const char* pope_status_string(int status) {
  switch (status) {
    case POPE_OK: return "ok";
    case POPE_ERR_INVALID_ARG: return "invalid argument";
    case POPE_ERR_DTYPE: return "unsupported dtype (POPE_F32 or POPE_BF16 only)";
    case POPE_ERR_WORKSPACE: return "workspace too small (see pope_coarse_workspace_bytes)";
    case POPE_ERR_SHAPE: return "shape not supported by the requested implementation";
    case POPE_ERR_ALIGNMENT: return "pointer or stride not sufficiently aligned";
    case POPE_ERR_CAPACITY: return "output capacity too small";
    case POPE_ERR_IO: return "file could not be created or written";
    default: return status > 0 ? cudaGetErrorString(static_cast<cudaError_t>(status)) : "unknown status";
  }
}

extern "C" int pope_coarse_auto_impl(int dtype, int L, int S, int C) {
  CoarseProblem p{};
  p.dtype = dtype; p.L = L; p.S = S; p.C = C; p.n = 1;
  p.log2_thr = -2.3219281f;      // thr = 0.2: fp32 features take the split tensor-core path at the default threshold
  return (coarse_tc_supported(p) || coarse_tc_split_supported(p)) ? POPE_COARSE_TCGEN05 : POPE_COARSE_SIMT;
}

extern "C" size_t pope_coarse_workspace_bytes(int n_pairs, int L, int S) {
  if (n_pairs <= 0 || L <= 0 || S <= 0) return 0;
  return carve_coarse_scratch(nullptr, n_pairs, L, S).bytes;
}

extern "C" size_t pope_coarse_workspace_bytes_ex(int n_pairs, int L, int S, int C, int dtype) {
  if (n_pairs <= 0 || L <= 0 || S <= 0 || C <= 0) return 0;
  size_t bytes = align_up(carve_coarse_scratch(nullptr, n_pairs, L, S).bytes, 256);
  if (dtype == POPE_F32 && C % 64 == 0 && C <= 256) bytes += coarse_tc_split_bytes(n_pairs, L, S, C);
  return bytes;
}

extern "C" int pope_coarse_match(const void* feat_c0, const void* feat_c1, int dtype, int n_pairs, int L, int S, int C,
                                 int h0c, int w0c, int h1c, int w1c, float pixel_scale, float temperature, float thr,
                                 int border_rm, int impl, void* workspace, size_t workspace_bytes, int64_t* b_ids,
                                 int64_t* i_ids, int64_t* j_ids, float* mconf, float* mkpts0_c, float* mkpts1_c,
                                 int32_t* counts, int64_t capacity, void* stream) {
  if (!feat_c0 || !feat_c1 || !workspace || !b_ids || !i_ids || !j_ids || !mconf || !mkpts0_c || !mkpts1_c || !counts)
    return POPE_ERR_INVALID_ARG;
  if (n_pairs <= 0 || n_pairs > 65535 || L <= 0 || S <= 0 || C <= 0) return POPE_ERR_INVALID_ARG;
  if (h0c <= 0 || w0c <= 0 || h1c <= 0 || w1c <= 0 || int64_t(h0c) * w0c != L || int64_t(h1c) * w1c != S)
    return POPE_ERR_INVALID_ARG;
  if (!(thr > 0.f) || !(thr <= 1.f) || !(temperature > 0.f) || border_rm < 0) return POPE_ERR_INVALID_ARG;
  if (dtype != POPE_F32 && dtype != POPE_BF16) return POPE_ERR_DTYPE;
  if (C % 16 != 0) return POPE_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(feat_c0) | reinterpret_cast<uintptr_t>(feat_c1) |
       reinterpret_cast<uintptr_t>(workspace)) & 15u)
    return POPE_ERR_ALIGNMENT;
  if (capacity < int64_t(n_pairs) * (L < S ? L : S)) return POPE_ERR_CAPACITY;
  CoarseScratch w = carve_coarse_scratch(workspace, n_pairs, L, S);
  if (workspace_bytes < w.bytes) return POPE_ERR_WORKSPACE;

  CoarseProblem p;
  p.f0 = feat_c0; p.f1 = feat_c1; p.dtype = dtype; p.n = n_pairs; p.L = L; p.S = S; p.C = C;
  p.h0c = h0c; p.w0c = w0c; p.h1c = h1c; p.w1c = w1c;
  // the reference divides both feature sets by sqrt(C) and the product by T (coarse_matching.py:109-114)
  p.scale_log2 = static_cast<float>(1.4426950408889634 / (double(C) * double(temperature)));
  p.log2_thr = static_cast<float>(log2(double(thr)));   // `conf > thr` is evaluated on fp32 values: thr arrives as float
  p.border = border_rm; p.pixel_scale = pixel_scale;

  // fp32 features: the tensor-core path splits every value into three bf16 terms (fp32 accuracy) and needs the larger
  // workspace of pope_coarse_workspace_bytes_ex; with the plain workspace (or thr <= 0.15, two_sweeps_possible) fp32 runs the fp32-FMA kernels
  const size_t std_bytes = align_up(w.bytes, 256);
  const bool split_ok = coarse_tc_split_supported(p) && workspace_bytes >= std_bytes + coarse_tc_split_bytes(n_pairs, L, S, C);
  bool use_tc, use_split = false;
  if (impl == POPE_COARSE_SIMT) use_tc = false;
  else if (impl == POPE_COARSE_TCGEN05) {
    if (coarse_tc_supported(p)) use_tc = true;
    else if (coarse_tc_split_supported(p)) { if (!split_ok) return POPE_ERR_WORKSPACE; use_tc = false; use_split = true; }
    else return POPE_ERR_SHAPE;
  }
  else if (impl == POPE_COARSE_AUTO) { use_tc = coarse_tc_supported(p); use_split = !use_tc && split_ok; }
  else return POPE_ERR_INVALID_ARG;

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  // clear the total/flag words (each launch sequence clears the scratch it needs cleared itself)
  if ((e = cudaMemsetAsync(counts + n_pairs, 0, 2 * sizeof(int32_t), st)) != cudaSuccess) return int(e);
  if (use_split) {
    // single sweep on the split planes, then the fp32-FMA kernels as a gated fallback (no-ops unless the flag was raised)
    e = coarse_tc_split_run(p, w, static_cast<char*>(workspace) + std_bytes, counts + n_pairs + 1, st);
    if (e == cudaSuccess) e = coarse_simt_run(p, w, counts + n_pairs + 1, st, true);
  } else {
    e = use_tc ? coarse_tc_run(p, w, counts + n_pairs + 1, st) : coarse_simt_run(p, w, counts + n_pairs + 1, st);
  }
  if (e != cudaSuccess) return int(e);
  e = coarse_finalize_run(p, w, b_ids, i_ids, j_ids, mconf, mkpts0_c, mkpts1_c, counts, capacity, st);
  return int(e);
}
