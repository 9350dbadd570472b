// Shared device-side types and helpers for libpnce (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pnce.h"

namespace pnce {

constexpr int kThreads = 256;          // every kernel in this library uses 256-thread CTAs
constexpr int kRowTile = 32;           // patches per gather / SIMT-loss CTA
constexpr int kTilePos = 2048;         // positions per tile of the dense backward (8 KB of fp32)
constexpr float kNormEps = 1e-6f;      // F.normalize eps               patchnce_cut.py:77-78
constexpr float kClamp = 50.0f;        // torch.clamp(logits, -50, 50)  patchnce_cut.py:88

// Per-layer view of the problem plus its slices of the caller's workspace.
struct LayerDev {
  const void* src;
  const void* tgt;
  void* dtgt;
  const long long* ids;
  int C, HW, P, nwords;      // nwords: unused (kept for layout stability)
  int ntiles;                // ceil(P / 32)
  int sorted;                // 1: rows / qinv are in sorted-slot order (tensor-core path), 0: ids order
  // id bookkeeping (written by the prep CTA of the gather launch)
  int* sid;                  // [P]   ids sorted ascending
  int* perm;                 // [P]   original index of sorted slot j
  int* rank;                 // [P]   sorted slot of original index p
  int* cslot;                // [ceil(HW/kTilePos)+1] first sorted slot whose id >= t * kTilePos
  // rows
  float* qn;                 // [B][P][C] normalised target rows (ids order)
  float* kn;                 // [B][P][C] normalised source rows
  float* qinv;               // [B][P]  +1/||x||, or -1/eps when ||x|| < eps, NaN for non-finite rows
  float* dxT;                // [B][C][dxpitch] d loss / d raw target patch, unit upstream, SORTED slot order
  int dxpitch;               // row pitch of dxT: P, or Ppad on the tensor-core path
  float* partial;            // [B][ntiles] partial sums of row losses
  float* dq_rows;            // optional [B][P][C] output of the rows API (then dxT/qinv unused)
  int nparts;                // partial row-loss sums per image (ntiles on the SIMT path, halves on TC)
  // ---- tensor-core path (gather_tc.cuh / loss_tc.cuh) ----
  int Cp, Ppad, nchunk;      // C rounded up to 32, P rounded up to 128 (<= 1024), Cp / 32
  __nv_bfloat16* qhi;        // Q operand blob, bf16 high part   [B][Ppad/128][Cp/8][16][8][8]
  __nv_bfloat16* qlo;        // low part (value - hi), NULL in single-pass bf16 mode
  __nv_bfloat16* khi;        // K operand blob, key blocks of <= 256  [B][kb][Cp/8][NB/8][8][8]
  __nv_bfloat16* klo;
  __nv_bfloat16* k2hi;       // the same K values, key-major  [B][Ppad/8][Cp/8][8][8]  (phase-2 B operand)
  __nv_bfloat16* k2lo;
  __nv_bfloat16* dyhi;       // head mode: d loss / d head output as a row blob (then dxT is not written)
  __nv_bfloat16* dylo;
  int head_src_rows;         // head mode gather: the src side is written as a row blob too (into khi/klo)
  float* qss;                // [B][nchunk][Ppad] partial sums of squares (NaN: non-finite element)
  float* kss;
  float* kinv;               // [B][Ppad] 1/max(||k_j||, eps) (0 for padding / non-finite rows), P > 256 only
};

struct Params {
  LayerDev L[PNCE_MAX_LAYERS];
  int n_layers, B, dtype, math;
  float tau;
  int side0;                 // first side the gather launch covers: 0 = src+tgt, 1 = tgt only
  int raw;                   // module-split API: 1 = rows are the raw patches (no L2 normalisation)
  int rows_mode;             // module-split rows API on the tensor-core kernel: rows are used as given (no
                             // normalisation, no normalise backward), d loss / d q leaves row-major in dq_rows
  int nhwc;                  // channels-last maps (nhwc.cuh): src/tgt/dtgt are (B, HW, C) storage and dxT holds ROW-major
                             // rows [image][sorted slot][C]; tensor-core path only
  int mb;                    // minibatch negatives (k_loss_tc_mb): each layer's B * P rows are ONE group (one CE mean,
                             // one non-finite guard) instead of B images
  int b0, bn;                // images [b0, b0+bn) of the batch are covered by this launch (chunked forward)
  unsigned total_ctas;       // loss CTAs over all chunks: the one that arrives last finalises
  float* loss_out;           // [1 + n_layers]
  int* nonfinite;            // [1]
  unsigned* counter;         // [1] last-CTA election; zeroed by the gather launch
  float* lossimg;            // [n_layers][B]
  int* valid;                // [n_layers][B]
  const float* grad_out;     // device scalar or NULL (=1)
  // ids drawn by the library (pnce_fwd_draw / pnce_plan_ids_draw): layer l's ids are what torch.randint(0, HW, (P,))
  // returns on a CUDA generator at (rng_seed, rng_offset + 4 l); k_prep writes them to L.ids before sorting them
  unsigned long long rng_seed, rng_offset;
  int rng_draw;
  long long* trace;          // debug: clock64 stamps of two CTAs of the tcgen05 loss kernel, or NULL
  // global negatives (pnce_mb_shard_loss; kworld = 0 otherwise): the key blobs of every layer (khi, klo, k2hi, k2lo,
  // kss) point into slot 0 of kworld slots of kslot bytes; slot w holds the keys of global images [w B, (w + 1) B).
  // This launch's query images are global images kimg0 + b.  qbad: slot 0's per-layer "a query row of that rank is
  // non-finite" flags (int[PNCE_MAX_LAYERS] at the head of every slot).
  int kworld, kimg0;
  size_t kslot;
  const int* qbad;
};

// CTA -> layer map for one launch: blocks [start[l], start[l+1]) work on layer l.
struct BlockMap {
  long long start[PNCE_MAX_LAYERS + 2];
  int layer[PNCE_MAX_LAYERS];          // slot -> layer (launch_loss_tc orders heavy layers first)
};

__device__ __forceinline__ int find_layer(const BlockMap& m, long long blk, int n) {
  int l = 0;
  for (int i = 1; i < n; ++i)
    if (blk >= m.start[i]) l = i;
  return l;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Programmatic dependent launch (griddepcontrol, sm_90+): FIRST statement of every kernel of this library except the
// dense-backward kernels, which are always launched the ordinary way (pnce_api.cu: launch_k, SITE 0).  The host
// launches the kernels of one step with cudaLaunchAttributeProgrammaticStreamSerialization (pnce_api.cu: launch_k), so
// the next kernel's CTAs are dispatched while this one drains and its launch latency is hidden; `wait` returns once
// every prerequisite grid has completed and its memory is visible, so nothing after it can see half-written data or
// overwrite what a predecessor still reads (every kernel waits before its first global access, which makes completion
// transitive along the stream).  Both instructions are no-ops for a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
// The tcgen05 kernels split the pair: pdl_launch() first, then their prologue -- mbarrier initialisation, TMEM allocation,
// the CTA-wide barrier: shared memory and TMEM only, 1-2 us per launch -- and pdl_wait() right behind it, still before the
// first global access; the prologue then runs under the predecessor's tail.  (A TMEM allocation that finds the columns
// still held by a predecessor's CTA on the same SM simply blocks until that CTA has exited.)
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// torch.clamp semantics: NaN propagates (fminf/fmaxf would swallow it).
__device__ __forceinline__ float clamp_nan(float x, float c) { return x < -c ? -c : (x > c ? c : x); }

}  // namespace pnce
