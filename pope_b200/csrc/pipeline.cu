// pipeline.cu -- the pair-batching driver behind pope_pipeline_* / pope_match_pairs_host.
//
// Replaces the batch-1 loop of the eval drivers (eval_linemod_json.py:103-122: three sequential matcher(batch)
// calls per test pair, each followed by three .cpu() syncs) by a chunked, double-buffered stream pipeline:
//   copy stream   : host -> device copies of chunk k+1
//   compute stream: [with a coarse level attached (pope_pipeline_set_coarse_level): position encoding of the chunk's
//                   backbone maps -> coarse transformer ->] coarse match -> fused window gather + fine match -> per-pair slotting of chunk k (no host sync:
//                   the match count stays on the device and gates the fine kernels); with a fine level attached
//                   (pope_pipeline_set_fine_level) coarse match -> window gather -> FinePreprocess Linears -> fine
//                   transformer -> fine match -> slotting, every launch bounded by the same device count
//   drain stream  : device -> host copies of chunk k-1
// One host synchronisation at the very end.
#include <new>
#include <stdlib.h>

#include "common.cuh"

namespace pope {
namespace {

// packed (sorted by pair) -> fixed per-pair slots, so that the host copy has a size known without a sync
__global__ void __launch_bounds__(256) slot_kernel(const int32_t* __restrict__ counts, int n_pairs, int cap,
                                                  const int64_t* __restrict__ i_ids, const int64_t* __restrict__ j_ids,
                                                  const float* __restrict__ mconf, const float* __restrict__ mk0,
                                                  const float* __restrict__ mk1f, int64_t* __restrict__ o_i,
                                                  int64_t* __restrict__ o_j, float* __restrict__ o_conf,
                                                  float* __restrict__ o_mk0, float* __restrict__ o_mk1) {
  __shared__ int s_base;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    int base = 0;
    for (int p = 0; p < b; ++p) base += counts[p];
    s_base = base;
  }
  __syncthreads();
  // (a pair can exceed its slot, and the packed list its capacity, only through bit-identical ties -- POPE_FLAG_CAPACITY)
  const int base = s_base, cnt = min(min(counts[b], cap), max(counts[n_pairs] - s_base, 0));
  for (int r = threadIdx.x; r < cnt; r += blockDim.x) {
    const size_t src = size_t(base) + r, dst = size_t(b) * cap + r;
    o_i[dst] = i_ids[src]; o_j[dst] = j_ids[src]; o_conf[dst] = mconf[src];
    reinterpret_cast<float2*>(o_mk0)[dst] = reinterpret_cast<const float2*>(mk0)[src];
    reinterpret_cast<float2*>(o_mk1)[dst] = reinterpret_cast<const float2*>(mk1f)[src];
  }
}

// ---- union fetch of the fine windows (image 1; with a fine level also image 0) ----------------------------------------
// The 5x5 windows of neighbouring matched cells overlap (window pitch = fine_stride < 5) and reads from page-locked host memory
// are not kept in L2, so fetching window by window moves the shared pixels once per window.  Instead the chunk's matched
// image-1 cells are marked in a byte map, and one kernel walks the fine map's pixels: a pixel that lies in the window of at
// least one marked cell is copied ONCE from the host buffer to the same place of the slot's device map, which the fused fine
// kernel then reads as after a bulk copy.  Bytes over the link: |union of the windows| <= min(sum of the windows, whole map).
__global__ void __launch_bounds__(256) mark_cells_kernel(const int32_t* __restrict__ total, int64_t capacity,
                                                        const int64_t* __restrict__ b_ids, const int64_t* __restrict__ j_ids,
                                                        int S, uint8_t* __restrict__ cellmask) {
  const int64_t M = min(int64_t(*total), capacity);
  for (int64_t m = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; m < M; m += int64_t(gridDim.x) * blockDim.x)
    cellmask[b_ids[m] * S + j_ids[m]] = 1;
}

__device__ __forceinline__ uint4 ld_host16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// 16-byte loads in flight per thread (4 / 8 / 16 and chunks of 4 / 8 / 16 / 32 pairs measured: 2 735-2 822 pairs/s, all within
// 3 %, best at 16 pairs per chunk -- the link, not the kernel's shape, sets the rate; profiles/r2_history.md)
constexpr int kFetchIt = 8;

// LPP = lanes (16-byte vectors) per pixel: 16 for 128 bf16 channels, 32 for fp32.  A warp owns kIt x (32 / LPP) consecutive
// pixels of the chunk's [n, Hf, Wf] map; all its loads are issued before the first store.
template <int LPP>
__global__ void __launch_bounds__(256) fetch_union_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst,
                                                         const uint8_t* __restrict__ cellmask, int64_t n_pix, int Hf, int Wf,
                                                         int hc, int wc, int stride, int half,
                                                         unsigned long long* __restrict__ fetched) {
  constexpr int PPI = 32 / LPP, kIt = kFetchIt;
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, sub = lane / LPP, v = lane % LPP;
  const int64_t warp = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t q0 = warp * (kIt * PPI);
  uint4 r[kIt];
  bool need[kIt];
#pragma unroll
  for (int k = 0; k < kIt; ++k) {
    const int64_t q = q0 + k * PPI + sub;
    need[k] = false;
    if (q < n_pix) {
      const int64_t b = q / (int64_t(Hf) * Wf);
      const int rem = int(q - b * (int64_t(Hf) * Wf));
      const int y = rem / Wf, x = rem - y * Wf;
      // cells c with c * stride - half <= y <= c * stride + half
      const int cy_lo = y > half ? (y - half + stride - 1) / stride : 0, cy_hi = min((y + half) / stride, hc - 1);
      const int cx_lo = x > half ? (x - half + stride - 1) / stride : 0, cx_hi = min((x + half) / stride, wc - 1);
      const uint8_t* cm = cellmask + b * (int64_t(hc) * wc);
      for (int cy = cy_lo; cy <= cy_hi; ++cy)
        for (int cx = cx_lo; cx <= cx_hi; ++cx) need[k] |= cm[cy * wc + cx] != 0;
    }
    if (need[k]) r[k] = ld_host16(src + (q * LPP + v));
  }
  int mine = 0;
#pragma unroll
  for (int k = 0; k < kIt; ++k) {
    if (need[k]) {
      dst[(q0 + k * PPI + sub) * LPP + v] = r[k];
      mine += v == 0;
    }
  }
  mine += __shfl_xor_sync(0xffffffffu, mine, 16);
  if (lane == 0 && mine) atomicAdd(&s_cnt, mine);
  __syncthreads();
  if (threadIdx.x == 0 && s_cnt) atomicAdd(fetched, (unsigned long long)s_cnt);
}

// the union fetch of one chunk's [n, Hf, Wf, Cf] fine map whose matched cells of the hc x wc grid are marked in cellmask
cudaError_t launch_fetch_union(const char* src, char* dst, const uint8_t* cellmask, int n, int Hf, int Wf, int hc, int wc,
                               int stride, int half, size_t pixel_bytes, unsigned long long* fetched, cudaStream_t st) {
  const int64_t np = int64_t(n) * Hf * Wf;
  const int lpp = int(pixel_bytes / 16), ppw = kFetchIt * (32 / lpp);                 // pixels per warp
  const unsigned blocks = unsigned((np + 8 * ppw - 1) / (8 * ppw));                   // 8 warps per block
  const uint4* s = reinterpret_cast<const uint4*>(src);
  uint4* d = reinterpret_cast<uint4*>(dst);
  if (lpp == 16)
    fetch_union_kernel<16><<<blocks, 256, 0, st>>>(s, d, cellmask, np, Hf, Wf, hc, wc, stride, half, fetched);
  else
    fetch_union_kernel<32><<<blocks, 256, 0, st>>>(s, d, cellmask, np, Hf, Wf, hc, wc, stride, half, fetched);
  return cudaGetLastError();
}

// default of POPE_PIPELINE_F1 for page-locked fine maps
constexpr bool kF1UnionDefault = true;

struct Slot {
  char *fc0 = nullptr, *fc1 = nullptr, *ff0 = nullptr, *ff1 = nullptr, *ws = nullptr;
  int64_t *b_ids = nullptr, *i_ids = nullptr, *j_ids = nullptr, *o_i = nullptr, *o_j = nullptr;
  float *mconf = nullptr, *mk0 = nullptr, *mk1 = nullptr, *expec = nullptr, *mk1f = nullptr, *o_conf = nullptr,
        *o_mk0 = nullptr, *o_mk1 = nullptr;
  int32_t* counts = nullptr;
  int32_t* h_counts = nullptr;   // pinned staging for the flag word
  uint8_t* cellmask = nullptr;   // [chunk, S] matched image-1 cells of the chunk (union fetch)
  char* maps = nullptr;          // with a coarse level: the chunk's fp32 backbone maps [chunk, C, L] | [chunk, C, S]
  cudaEvent_t uploaded = nullptr, computed = nullptr, drained = nullptr;
};

}  // namespace
}  // namespace pope

using namespace pope;

struct pope_pipeline {
  int device, dtype, chunk, C, Cf, h0c, w0c, h1c, w1c, fstride, W, L, S, cap, esize, impl, border;
  float pixel_scale, fine_scale, temperature, thr;
  size_t ws_bytes;
  int last_f1_mode = 0;            // how image 1's fine map reached the device in the last run: 0 bulk, 1 windows in place, 2 union fetch
  int64_t last_h2d_bytes = 0;      // bytes that crossed the host link towards the device in the last run
  cudaStream_t s_copy = nullptr, s_comp = nullptr, s_drain = nullptr;
  unsigned long long* fetched = nullptr;     // device: pixels of the fine maps the union fetch has copied in this run
  unsigned long long* h_fetched = nullptr;   // pinned staging for it
  Slot slot[2];
  // the fine level (pope_pipeline_set_fine_level_ex, in the pipeline's dtype): caller-owned packed weights; windows, image 0's cell mask and
  // scratch are allocated on the first attach and shared by both slots (all of it is touched on s_comp only)
  const void* fine_pre = nullptr;
  const void* fine_layers = nullptr;
  int fine_n_layers = 0;
  int* fine_kinds = nullptr;                 // host copy of layer_kinds
  char *win0 = nullptr, *win1 = nullptr, *fine_ws = nullptr;
  size_t fine_ws_bytes = 0;
  uint8_t* cellmask0 = nullptr;              // [chunk, L] matched image-0 cells of the chunk (union fetch of image 0)
  // the coarse level (pope_pipeline_set_coarse_level, in the pipeline's dtype): caller-owned encoding and packed layers;
  // each slot's map staging buffer (Slot::maps) and one transformer scratch shared by both slots (touched on s_comp only)
  // are allocated on the first attach
  const void* coarse_pe = nullptr;
  int pe_h = 0, pe_w = 0;
  const void* coarse_layers = nullptr;
  int coarse_n_layers = 0;
  int* coarse_kinds = nullptr;               // host copy of layer_kinds
  char* coarse_ws = nullptr;
  size_t coarse_ws_bytes = 0;
};

#define PL_CUDA(x)                                   \
  do {                                               \
    cudaError_t e__ = (x);                           \
    if (e__ != cudaSuccess) { rc = int(e__); goto fail; } \
  } while (0)

extern "C" int pope_pipeline_destroy(pope_pipeline_t* pl) {
  if (!pl) return POPE_OK;
  cudaSetDevice(pl->device);
  for (Slot& s : pl->slot) {
    void* bufs[] = {s.fc0, s.fc1, s.ff0, s.ff1, s.ws, s.b_ids, s.i_ids, s.j_ids, s.o_i, s.o_j, s.mconf,
                    s.mk0, s.mk1, s.expec, s.mk1f, s.o_conf, s.o_mk0, s.o_mk1, s.counts, s.cellmask, s.maps};
    for (void* b : bufs) if (b) cudaFree(b);
    if (s.h_counts) cudaFreeHost(s.h_counts);
    if (s.uploaded) cudaEventDestroy(s.uploaded);
    if (s.computed) cudaEventDestroy(s.computed);
    if (s.drained) cudaEventDestroy(s.drained);
  }
  if (pl->fetched) cudaFree(pl->fetched);
  if (pl->h_fetched) cudaFreeHost(pl->h_fetched);
  void* fine_bufs[] = {pl->win0, pl->win1, pl->fine_ws, pl->cellmask0, pl->coarse_ws};
  for (void* b : fine_bufs) if (b) cudaFree(b);
  free(pl->fine_kinds);
  free(pl->coarse_kinds);
  if (pl->s_copy) cudaStreamDestroy(pl->s_copy);
  if (pl->s_comp) cudaStreamDestroy(pl->s_comp);
  if (pl->s_drain) cudaStreamDestroy(pl->s_drain);
  delete pl;
  return POPE_OK;
}

extern "C" int pope_pipeline_create(pope_pipeline_t** out, int device, int dtype, int chunk_pairs, int C, int Cf, int h0c,
                                    int w0c, int h1c, int w1c, int fine_stride, int W, float pixel_scale,
                                    float fine_scale, float temperature, float thr, int border_rm, int impl) {
  if (!out) return POPE_ERR_INVALID_ARG;
  *out = nullptr;
  if (dtype != POPE_F32 && dtype != POPE_BF16) return POPE_ERR_DTYPE;
  if (chunk_pairs <= 0 || C <= 0 || Cf <= 0 || h0c <= 0 || w0c <= 0 || h1c <= 0 || w1c <= 0 || fine_stride <= 0 || W <= 0)
    return POPE_ERR_INVALID_ARG;
  if (Cf != 128 || W != 5) return POPE_ERR_SHAPE;
  int rc = POPE_OK;
  pope_pipeline* pl = new (std::nothrow) pope_pipeline();
  if (!pl) return int(cudaErrorMemoryAllocation);
  pl->device = device; pl->dtype = dtype; pl->chunk = chunk_pairs; pl->C = C; pl->Cf = Cf;
  pl->h0c = h0c; pl->w0c = w0c; pl->h1c = h1c; pl->w1c = w1c; pl->fstride = fine_stride; pl->W = W;
  pl->L = h0c * w0c; pl->S = h1c * w1c; pl->cap = pl->L < pl->S ? pl->L : pl->S;
  pl->esize = dtype == POPE_BF16 ? 2 : 4; pl->impl = impl; pl->border = border_rm;
  pl->pixel_scale = pixel_scale; pl->fine_scale = fine_scale; pl->temperature = temperature; pl->thr = thr;
  // (for fp32 features the larger size lets the coarse stage run on the tensor cores, see pope_b200.h)
  pl->ws_bytes = impl == POPE_COARSE_SIMT ? pope_coarse_workspace_bytes(chunk_pairs, pl->L, pl->S)
                                          : pope_coarse_workspace_bytes_ex(chunk_pairs, pl->L, pl->S, C, dtype);
  {
    const size_t n = chunk_pairs, e = pl->esize, capt = n * pl->cap;
    const size_t f0px = size_t(h0c) * fine_stride * w0c * fine_stride, f1px = size_t(h1c) * fine_stride * w1c * fine_stride;
    PL_CUDA(cudaSetDevice(device));
    PL_CUDA(cudaStreamCreateWithFlags(&pl->s_copy, cudaStreamNonBlocking));
    PL_CUDA(cudaStreamCreateWithFlags(&pl->s_comp, cudaStreamNonBlocking));
    PL_CUDA(cudaStreamCreateWithFlags(&pl->s_drain, cudaStreamNonBlocking));
    PL_CUDA(cudaMalloc(&pl->fetched, 8));
    PL_CUDA(cudaMallocHost(&pl->h_fetched, 8));
    for (Slot& s : pl->slot) {
      PL_CUDA(cudaMalloc(&s.cellmask, n * pl->S));
      PL_CUDA(cudaMalloc(&s.fc0, n * pl->L * C * e));
      PL_CUDA(cudaMalloc(&s.fc1, n * pl->S * C * e));
      PL_CUDA(cudaMalloc(&s.ff0, n * f0px * Cf * e));
      PL_CUDA(cudaMalloc(&s.ff1, n * f1px * Cf * e));
      PL_CUDA(cudaMalloc(&s.ws, pl->ws_bytes));
      PL_CUDA(cudaMalloc(&s.b_ids, capt * 8)); PL_CUDA(cudaMalloc(&s.i_ids, capt * 8)); PL_CUDA(cudaMalloc(&s.j_ids, capt * 8));
      PL_CUDA(cudaMalloc(&s.o_i, capt * 8)); PL_CUDA(cudaMalloc(&s.o_j, capt * 8));
      PL_CUDA(cudaMalloc(&s.mconf, capt * 4)); PL_CUDA(cudaMalloc(&s.o_conf, capt * 4));
      PL_CUDA(cudaMalloc(&s.mk0, capt * 8)); PL_CUDA(cudaMalloc(&s.mk1, capt * 8)); PL_CUDA(cudaMalloc(&s.mk1f, capt * 8));
      PL_CUDA(cudaMalloc(&s.o_mk0, capt * 8)); PL_CUDA(cudaMalloc(&s.o_mk1, capt * 8));
      PL_CUDA(cudaMalloc(&s.expec, capt * 12));
      PL_CUDA(cudaMalloc(&s.counts, (n + 2) * 4));
      PL_CUDA(cudaMallocHost(&s.h_counts, (n + 2) * 4));
      PL_CUDA(cudaEventCreateWithFlags(&s.uploaded, cudaEventDisableTiming));
      PL_CUDA(cudaEventCreateWithFlags(&s.computed, cudaEventDisableTiming));
      PL_CUDA(cudaEventCreateWithFlags(&s.drained, cudaEventDisableTiming));
    }
  }
  *out = pl;
  return POPE_OK;
fail:
  pope_pipeline_destroy(pl);
  return rc;
}

extern "C" int pope_pipeline_set_fine_level_ex(pope_pipeline_t* pl, int dtype, const void* pre, const void* layers,
                                               int n_layers, const int* layer_kinds) {
  if (!pl) return POPE_ERR_INVALID_ARG;
  if (!layers) {                 // detach; the windows and scratch stay allocated until pope_pipeline_destroy
    pl->fine_pre = pl->fine_layers = nullptr;
    pl->fine_n_layers = 0;
    return POPE_OK;
  }
  if (n_layers < 1 || !layer_kinds) return POPE_ERR_INVALID_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (layer_kinds[l] != 0 && layer_kinds[l] != 1) return POPE_ERR_INVALID_ARG;
  if (dtype != pl->dtype) return POPE_ERR_DTYPE;
  if (pl->C != 256) return POPE_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(pre) | reinterpret_cast<uintptr_t>(layers)) & 15u) return POPE_ERR_ALIGNMENT;
  int rc = POPE_OK;
  int* kinds = static_cast<int*>(malloc(sizeof(int) * size_t(n_layers)));
  if (!kinds) return int(cudaErrorMemoryAllocation);
  for (int l = 0; l < n_layers; ++l) kinds[l] = layer_kinds[l];
  if (!pl->win0) {
    // sized by the chunk's capacity, like every other slot buffer: the launches are bounded by the device count; the
    // windows have the pipeline's element type
    const int64_t m = int64_t(pl->chunk) * pl->cap;
    const int ww = pl->W * pl->W;
    const size_t win_bytes = size_t(m) * ww * pl->Cf * pl->esize;
    const bool f32 = pl->dtype == POPE_F32;
    const size_t tf = f32 ? pope_fine_tf_f32_workspace_bytes(m, ww) : pope_fine_tf_workspace_bytes(m, ww);
    const size_t mg = f32 ? pope_fine_merge_f32_workspace_bytes(m) : pope_fine_merge_workspace_bytes(m);
    PL_CUDA(cudaSetDevice(pl->device));
    PL_CUDA(cudaMalloc(&pl->win0, win_bytes));
    PL_CUDA(cudaMalloc(&pl->win1, win_bytes));
    PL_CUDA(cudaMalloc(&pl->fine_ws, tf > mg ? tf : mg));
    PL_CUDA(cudaMalloc(&pl->cellmask0, size_t(pl->chunk) * pl->L));
    pl->fine_ws_bytes = tf > mg ? tf : mg;
  }
  free(pl->fine_kinds);
  pl->fine_kinds = kinds;
  pl->fine_pre = pre;
  pl->fine_layers = layers;
  pl->fine_n_layers = n_layers;
  return POPE_OK;
fail:
  free(kinds);
  cudaFree(pl->win0); cudaFree(pl->win1); cudaFree(pl->fine_ws); cudaFree(pl->cellmask0);   // (cudaFree(NULL) is a no-op)
  pl->win0 = pl->win1 = pl->fine_ws = nullptr;
  pl->cellmask0 = nullptr;
  return rc;
}

extern "C" int pope_pipeline_set_fine_level(pope_pipeline_t* pl, const void* pre, const void* layers, int n_layers,
                                            const int* layer_kinds) {
  return pope_pipeline_set_fine_level_ex(pl, POPE_BF16, pre, layers, n_layers, layer_kinds);
}

extern "C" int pope_pipeline_set_coarse_level(pope_pipeline_t* pl, int dtype, const void* pe, int pe_h, int pe_w,
                                              const void* layers, int n_layers, const int* layer_kinds) {
  if (!pl) return POPE_ERR_INVALID_ARG;
  if (!layers) {                 // detach; the staging buffers and scratch stay allocated until pope_pipeline_destroy
    pl->coarse_pe = pl->coarse_layers = nullptr;
    pl->coarse_n_layers = 0;
    return POPE_OK;
  }
  if (!pe || pe_h <= 0 || pe_w <= 0 || n_layers < 1 || !layer_kinds) return POPE_ERR_INVALID_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (layer_kinds[l] != 0 && layer_kinds[l] != 1) return POPE_ERR_INVALID_ARG;
  if (dtype != pl->dtype) return POPE_ERR_DTYPE;
  if (pl->C != 256 || pl->h0c > pe_h || pl->w0c > pe_w || pl->h1c > pe_h || pl->w1c > pe_w) return POPE_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(pe) & 3u) || (reinterpret_cast<uintptr_t>(layers) & 15u)) return POPE_ERR_ALIGNMENT;
  const bool f32 = pl->dtype == POPE_F32;
  const size_t tf = f32 ? pope_coarse_tf_f32_workspace_bytes(pl->chunk, pl->L, pl->S)
                        : pope_coarse_tf_workspace_bytes(pl->chunk, pl->L, pl->S);
  if (tf == 0) return POPE_ERR_SHAPE;
  int rc = POPE_OK;
  int* kinds = static_cast<int*>(malloc(sizeof(int) * size_t(n_layers)));
  if (!kinds) return int(cudaErrorMemoryAllocation);
  for (int l = 0; l < n_layers; ++l) kinds[l] = layer_kinds[l];
  if (!pl->coarse_ws) {
    // the maps cross the link in fp32 whatever the pipeline's dtype: the encoding is added in fp32 before any rounding
    const size_t map_bytes = size_t(pl->chunk) * (pl->L + pl->S) * pl->C * sizeof(float);
    PL_CUDA(cudaSetDevice(pl->device));
    for (Slot& s : pl->slot) PL_CUDA(cudaMalloc(&s.maps, map_bytes));
    PL_CUDA(cudaMalloc(&pl->coarse_ws, tf));
    pl->coarse_ws_bytes = tf;
  }
  free(pl->coarse_kinds);
  pl->coarse_kinds = kinds;
  pl->coarse_pe = pe;
  pl->pe_h = pe_h;
  pl->pe_w = pe_w;
  pl->coarse_layers = layers;
  pl->coarse_n_layers = n_layers;
  return POPE_OK;
fail:
  free(kinds);
  for (Slot& s : pl->slot) { cudaFree(s.maps); s.maps = nullptr; }     // (cudaFree(NULL) is a no-op)
  cudaFree(pl->coarse_ws);
  pl->coarse_ws = nullptr;
  return rc;
}

extern "C" int pope_pipeline_run(pope_pipeline_t* pl, const void* feat_c0, const void* feat_c1, const void* feat_f0,
                                 const void* feat_f1, int n_pairs, int64_t* i_ids, int64_t* j_ids, float* mconf,
                                 float* mkpts0_f, float* mkpts1_f, int32_t* counts, int32_t* flags) {
  if (!pl || !feat_c0 || !feat_c1 || !feat_f0 || !feat_f1 || !i_ids || !j_ids || !mconf || !mkpts0_f || !mkpts1_f ||
      !counts || n_pairs <= 0)
    return POPE_ERR_INVALID_ARG;
  int rc = POPE_OK;
  const size_t e = pl->esize, L = pl->L, S = pl->S, C = pl->C, Cf = pl->Cf, cap = pl->cap;
  const int Hf0 = pl->h0c * pl->fstride, Wf0 = pl->w0c * pl->fstride, Hf1 = pl->h1c * pl->fstride, Wf1 = pl->w1c * pl->fstride;
  const size_t fc0_pair = L * C * e, fc1_pair = S * C * e, ff0_pair = size_t(Hf0) * Wf0 * Cf * e,
               ff1_pair = size_t(Hf1) * Wf1 * Cf * e;
  // channels-last element strides (n, c, h, w) of the device copies
  const int64_t st0[4] = {int64_t(Hf0) * Wf0 * int64_t(Cf), 1, int64_t(Wf0) * int64_t(Cf), int64_t(Cf)};
  const int64_t st1[4] = {int64_t(Hf1) * Wf1 * int64_t(Cf), 1, int64_t(Wf1) * int64_t(Cf), int64_t(Cf)};
  const float coord_scale = float(pl->W / 2) * pl->fine_scale;
  // Without a fine level, of image 0's fine map the pipeline only ever reads the centre pixel of each MATCHED cell (window
  // 0 contributes its centre row to the fine correlation, fine_matching.py:43).  When the caller's buffer is page-locked (device-
  // addressable under UVA) the fused fine kernel fetches those pixels straight from host memory (M x 256 B per chunk
  // instead of copying the whole 1/2-resolution map); pageable buffers fall back to the bulk copy.
  const char* f0_dev_view = nullptr;
  const char* f1_dev_view = nullptr;
  auto host_view = [](const void* p) -> const char* {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
      return static_cast<const char*>(attr.devicePointer);
    cudaGetLastError();   // clear the "invalid value" some drivers report for pageable pointers
    return nullptr;
  };
  f0_dev_view = host_view(feat_f0);
  // Of image 1's map only the 5x5 windows of the matched cells are needed.  When its buffer is page-locked there are three
  // ways to get them, POPE_PIPELINE_F1 in the environment (measured on 64 pairs at 480x640, one B200, profiles/r2_history.md):
  //   union   (default): the union of the windows is fetched once per pixel into the slot's device map (fetch_union_kernel
  //                      above) and the fine kernel reads the device map -- 12.5 MB per pair, 2 820 pairs/s end to end;
  //   windows          : the fine kernel reads window by window in place over the link (M x 25 x 256 B = 16.3 MB per pair at
  //                      2 544 matches: pixels shared by neighbouring windows cross the link twice) -- 2 269 pairs/s;
  //   bulk (or POPE_PIPELINE_WINDOWS_IN_PLACE=0): the whole 19.7 MB map is copied -- 2 163 pairs/s.
  bool f1_union = kF1UnionDefault;
  {
    const char* env = getenv("POPE_PIPELINE_WINDOWS_IN_PLACE");
    const char* mode = getenv("POPE_PIPELINE_F1");
    bool bulk = env && env[0] == '0';
    if (mode && mode[0] == 'u') f1_union = true;
    if (mode && mode[0] == 'w') f1_union = false;
    if (mode && mode[0] == 'b') bulk = true;
    if (!bulk) f1_dev_view = host_view(feat_f1);
    if (!f1_dev_view || (Cf * e != 256 && Cf * e != 512)) f1_union = false;
  }
  // With a fine level the transformer needs all W*W pixels of image 0's windows, not only their centres, so image 0 takes
  // the form chosen for image 1: its windows' union is fetched into the slot's device map, the gather reads its windows in
  // place, or (image 1 copied whole, or a pageable image-0 buffer) the whole map is copied.  (f0_union implies f1_union.)
  const bool fine = pl->fine_layers != nullptr;
  if (fine && !f1_dev_view) f0_dev_view = nullptr;
  // With a coarse level, feat_c0 / feat_c1 are the backbone's fp32 maps [n, C, h, w]: they are staged in the slot and turned
  // into the token-major transformed features s.fc0 / s.fc1 on the compute stream.
  const bool coarse = pl->coarse_layers != nullptr;
  const size_t in_c0_pair = coarse ? L * C * sizeof(float) : fc0_pair, in_c1_pair = coarse ? S * C * sizeof(float) : fc1_pair;
  const bool f0_union = fine && f1_union && f0_dev_view;
  int64_t h2d = 0;
  int32_t flag_acc = 0;
  int n_chunks = (n_pairs + pl->chunk - 1) / pl->chunk;
  PL_CUDA(cudaSetDevice(pl->device));
  if (f1_union) PL_CUDA(cudaMemsetAsync(pl->fetched, 0, 8, pl->s_comp));
  for (int k = 0; k < n_chunks; ++k) {
    Slot& s = pl->slot[k & 1];
    const int p0 = k * pl->chunk, n = (n_pairs - p0 < pl->chunk) ? n_pairs - p0 : pl->chunk;
    const size_t capt = size_t(n) * cap;
    if (k >= 2) {
      // the slot's previous results must have left the device before its inputs/outputs are overwritten
      PL_CUDA(cudaStreamWaitEvent(pl->s_copy, s.computed, 0));
      PL_CUDA(cudaStreamWaitEvent(pl->s_comp, s.drained, 0));
      PL_CUDA(cudaEventSynchronize(s.drained));
      flag_acc |= s.h_counts[pl->chunk + 1];
    }
    char* dc0 = coarse ? s.maps : s.fc0;
    char* dc1 = coarse ? s.maps + size_t(pl->chunk) * in_c0_pair : s.fc1;
    PL_CUDA(cudaMemcpyAsync(dc0, static_cast<const char*>(feat_c0) + p0 * in_c0_pair, n * in_c0_pair, cudaMemcpyHostToDevice, pl->s_copy));
    PL_CUDA(cudaMemcpyAsync(dc1, static_cast<const char*>(feat_c1) + p0 * in_c1_pair, n * in_c1_pair, cudaMemcpyHostToDevice, pl->s_copy));
    if (!f0_dev_view)
      PL_CUDA(cudaMemcpyAsync(s.ff0, static_cast<const char*>(feat_f0) + p0 * ff0_pair, n * ff0_pair, cudaMemcpyHostToDevice, pl->s_copy));
    h2d += int64_t(n) * int64_t(in_c0_pair + in_c1_pair + (f1_dev_view ? 0 : ff1_pair) + (f0_dev_view ? 0 : ff0_pair));
    if (!f1_dev_view)
      PL_CUDA(cudaMemcpyAsync(s.ff1, static_cast<const char*>(feat_f1) + p0 * ff1_pair, n * ff1_pair, cudaMemcpyHostToDevice, pl->s_copy));
    PL_CUDA(cudaEventRecord(s.uploaded, pl->s_copy));
    PL_CUDA(cudaStreamWaitEvent(pl->s_comp, s.uploaded, 0));
    if (coarse) {
      rc = pope_coarse_pos_encode_ex(dc0, pl->coarse_pe, n, int(C), pl->h0c, pl->w0c, pl->pe_h, pl->pe_w, s.fc0, pl->dtype,
                                     pl->s_comp);
      if (rc) goto fail;
      rc = pope_coarse_pos_encode_ex(dc1, pl->coarse_pe, n, int(C), pl->h1c, pl->w1c, pl->pe_h, pl->pe_w, s.fc1, pl->dtype,
                                     pl->s_comp);
      if (rc) goto fail;
      rc = (pl->dtype == POPE_F32 ? pope_coarse_transformer_f32 : pope_coarse_transformer)(
          s.fc0, s.fc1, n, pl->L, pl->S, pl->coarse_layers, pl->coarse_n_layers, pl->coarse_kinds, pl->coarse_ws,
          pl->coarse_ws_bytes, pl->s_comp);
      if (rc) goto fail;
    }
    rc = pope_coarse_match(s.fc0, s.fc1, pl->dtype, n, pl->L, pl->S, pl->C, pl->h0c, pl->w0c, pl->h1c, pl->w1c,
                           pl->pixel_scale, pl->temperature, pl->thr, pl->border, pl->impl, s.ws, pl->ws_bytes, s.b_ids,
                           s.i_ids, s.j_ids, s.mconf, s.mk0, s.mk1, s.counts, int64_t(capt), pl->s_comp);
    if (rc) goto fail;
    if (f1_union) {
      PL_CUDA(cudaMemsetAsync(s.cellmask, 0, size_t(n) * S, pl->s_comp));
      mark_cells_kernel<<<64, 256, 0, pl->s_comp>>>(s.counts + n, int64_t(capt), s.b_ids, s.j_ids, int(S), s.cellmask);
      PL_CUDA(launch_fetch_union(f1_dev_view + p0 * ff1_pair, s.ff1, s.cellmask, n, Hf1, Wf1, pl->h1c, pl->w1c, pl->fstride,
                                 pl->W / 2, Cf * e, pl->fetched, pl->s_comp));
    }
    if (f0_union) {
      PL_CUDA(cudaMemsetAsync(pl->cellmask0, 0, size_t(n) * L, pl->s_comp));
      mark_cells_kernel<<<64, 256, 0, pl->s_comp>>>(s.counts + n, int64_t(capt), s.b_ids, s.i_ids, int(L), pl->cellmask0);
      PL_CUDA(launch_fetch_union(f0_dev_view + p0 * ff0_pair, s.ff0, pl->cellmask0, n, Hf0, Wf0, pl->h0c, pl->w0c, pl->fstride,
                                 pl->W / 2, Cf * e, pl->fetched, pl->s_comp));
    }
    if (fine) {
      // gather -> [down_proj / merge_feat] -> encoder layers -> fine match on the windows, all bounded by the chunk's count
      const int64_t m = int64_t(capt);
      const int32_t* m_dev = s.counts + n;
      const int ww = pl->W * pl->W;
      rc = pope_fine_gather((f0_dev_view && !f0_union) ? static_cast<const void*>(f0_dev_view + p0 * ff0_pair) : s.ff0,
                            (f1_dev_view && !f1_union) ? static_cast<const void*>(f1_dev_view + p0 * ff1_pair) : s.ff1,
                            pl->dtype, n, pl->Cf, Hf0, Wf0, st0, Hf1, Wf1, st1, pl->w0c, pl->w1c, pl->fstride, pl->W, s.b_ids,
                            s.i_ids, s.j_ids, m, m_dev, pl->win0, pl->win1, pl->s_comp);
      if (rc) goto fail;
      const bool f32 = pl->dtype == POPE_F32;
      if (pl->fine_pre) {
        rc = (f32 ? pope_fine_merge_coarse_f32_ex : pope_fine_merge_coarse_ex)(
            pl->win0, pl->win1, m, m_dev, ww, s.fc0, s.fc1, pl->L, pl->S, pl->C, s.b_ids, s.i_ids, s.j_ids, pl->fine_pre,
            pl->fine_ws, pl->fine_ws_bytes, pl->s_comp);
        if (rc) goto fail;
      }
      rc = (f32 ? pope_fine_transformer_f32_ex : pope_fine_transformer_ex)(pl->win0, pl->win1, m, m_dev, ww, pl->fine_layers,
                                                                           pl->fine_n_layers, pl->fine_kinds, pl->fine_ws,
                                                                           pl->fine_ws_bytes, pl->s_comp);
      if (rc) goto fail;
      rc = pope_fine_match(pl->win0, pl->win1, pl->dtype, m, m_dev, ww, pl->Cf, s.mk1, coord_scale, s.expec, s.mk1f,
                           pl->s_comp);
      if (rc) goto fail;
    } else {
      rc = pope_fine_match_maps(f0_dev_view ? static_cast<const void*>(f0_dev_view + p0 * ff0_pair) : s.ff0,
                                (f1_dev_view && !f1_union) ? static_cast<const void*>(f1_dev_view + p0 * ff1_pair) : s.ff1, pl->dtype, n, pl->Cf, Hf0, Wf0, st0, Hf1, Wf1, st1, pl->w0c, pl->w1c,
                                pl->fstride, pl->W, s.b_ids, s.i_ids, s.j_ids, int64_t(capt), s.counts + n, nullptr, s.mk1,
                                coord_scale, s.expec, s.mk1f, pl->s_comp);
      if (rc) goto fail;
    }
    slot_kernel<<<n, 256, 0, pl->s_comp>>>(s.counts, n, int(cap), s.i_ids, s.j_ids, s.mconf, s.mk0, s.mk1f, s.o_i, s.o_j,
                                           s.o_conf, s.o_mk0, s.o_mk1);
    PL_CUDA(cudaGetLastError());
    PL_CUDA(cudaEventRecord(s.computed, pl->s_comp));
    PL_CUDA(cudaStreamWaitEvent(pl->s_drain, s.computed, 0));
    PL_CUDA(cudaMemcpyAsync(i_ids + size_t(p0) * cap, s.o_i, capt * 8, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(j_ids + size_t(p0) * cap, s.o_j, capt * 8, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(mconf + size_t(p0) * cap, s.o_conf, capt * 4, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(mkpts0_f + size_t(p0) * cap * 2, s.o_mk0, capt * 8, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(mkpts1_f + size_t(p0) * cap * 2, s.o_mk1, capt * 8, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(counts + p0, s.counts, size_t(n) * 4, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaMemcpyAsync(s.h_counts + pl->chunk + 1, s.counts + n + 1, 4, cudaMemcpyDeviceToHost, pl->s_drain));
    PL_CUDA(cudaEventRecord(s.drained, pl->s_drain));
  }
  if (f1_union) PL_CUDA(cudaMemcpyAsync(pl->h_fetched, pl->fetched, 8, cudaMemcpyDeviceToHost, pl->s_drain));   // (behind the last chunk's drain)
  PL_CUDA(cudaStreamSynchronize(pl->s_drain));
  for (int k = (n_chunks >= 2 ? n_chunks - 2 : 0); k < n_chunks; ++k) flag_acc |= pl->slot[k & 1].h_counts[pl->chunk + 1];
  if (flags) *flags = flag_acc;
  if (f0_dev_view || (f1_dev_view && !f1_union)) {   // what the fine kernel read in place also crossed the host link
    int64_t m = 0;
    for (int p = 0; p < n_pairs; ++p) m += counts[p];
    if (f0_dev_view && !fine) h2d += m * int64_t(Cf * e);                                    // image 0: the centre pixels
    if (f0_dev_view && fine && !f0_union) h2d += m * int64_t(pl->W * pl->W) * int64_t(Cf * e);   // image 0: every window whole
    if (f1_dev_view && !f1_union) h2d += m * int64_t(pl->W * pl->W) * int64_t(Cf * e);       // image 1: every window whole
  }
  if (f1_union) h2d += int64_t(*pl->h_fetched) * int64_t(Cf * e);   // every pixel of the windows' union(s) exactly once
  pl->last_f1_mode = f1_union ? 2 : f1_dev_view ? 1 : 0;
  pl->last_h2d_bytes = h2d;
  return POPE_OK;
fail:
  cudaStreamSynchronize(pl->s_copy); cudaStreamSynchronize(pl->s_comp); cudaStreamSynchronize(pl->s_drain);
  return rc;
}

extern "C" int pope_match_pairs_host(const void* feat_c0, const void* feat_c1, const void* feat_f0, const void* feat_f1,
                                     int dtype, int n_pairs, int C, int Cf, int h0c, int w0c, int h1c, int w1c,
                                     int fine_stride, int W, float pixel_scale, float fine_scale, float temperature,
                                     float thr, int border_rm, int impl, int chunk_pairs, int device, int64_t* i_ids,
                                     int64_t* j_ids, float* mconf, float* mkpts0_f, float* mkpts1_f, int32_t* counts,
                                     int32_t* flags) {
  if (n_pairs <= 0) return POPE_ERR_INVALID_ARG;
  if (chunk_pairs <= 0) chunk_pairs = n_pairs < 16 ? n_pairs : 16;
  if (chunk_pairs > n_pairs) chunk_pairs = n_pairs;
  pope_pipeline_t* pl = nullptr;
  int rc = pope_pipeline_create(&pl, device, dtype, chunk_pairs, C, Cf, h0c, w0c, h1c, w1c, fine_stride, W, pixel_scale,
                                fine_scale, temperature, thr, border_rm, impl);
  if (rc) return rc;
  rc = pope_pipeline_run(pl, feat_c0, feat_c1, feat_f0, feat_f1, n_pairs, i_ids, j_ids, mconf, mkpts0_f, mkpts1_f, counts,
                         flags);
  pope_pipeline_destroy(pl);
  return rc;
}

extern "C" int64_t pope_pipeline_last_h2d_bytes(const pope_pipeline_t* pl) { return pl ? pl->last_h2d_bytes : 0; }
extern "C" int pope_pipeline_last_f1_mode(const pope_pipeline_t* pl) { return pl ? pl->last_f1_mode : -1; }
