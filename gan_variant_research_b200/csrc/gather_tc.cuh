// Tensor-core path, launch 2 (after k_prep): random-patch gather that writes the MMA operands directly.
//   CTA  <-> (layer, side, image, chunk of 32 channels);  thread <-> sorted slot p  (P <= 256):
//   row p of every operand is the patch with the p-th smallest id (k_prep's sid[]), see loss_tc.cuh
//   every thread issues 32 independent L2-only loads (one sector each: element (c, id) of an NCHW
//   plane), splits each value into bf16 hi + lo, and stores 8 consecutive channels as one 16-byte
//   row of an 8x8 core matrix.  The global operand blobs are laid out exactly as the shared-memory
//   image the tensor core reads (no-swizzle canonical layout), so the loss kernel moves them with
//   1-D bulk copies:
//     Q blob: [image][half m = p/128][c/8][16 row groups][8 rows][8 ch]   bf16
//     K blob: [image][c/8][Ppad/8 row groups][8 rows][8 ch]                bf16
//   Values are RAW (not normalised): the row norms are only known once all channels are seen, so
//   each chunk also emits its partial sum of squares and the loss kernel folds 1/||q||, 1/||k||
//   into its epilogues (the normalise backward re-reads the raw q values as hi + lo from the Q blob).
//   Replaces patchnce_cut.py:56-78 on the tensor-core path.
#pragma once
#include "common.cuh"
#include "gather.cuh"

namespace pnce {

__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// keys_s != NULL (k_gather_tc_fold): the layer's sorted (id, index) keys are in shared memory, sid[] is not read
template <typename T>
__device__ void gather_tc_chunk(const LayerDev& L, int b0, int B, long long local, int side0,
                                const unsigned long long* keys_s = nullptr) {
  const int nchunk = L.nchunk;
  const int npb = (L.Ppad + 255) >> 8;                       // CTAs of 256 patch slots per (image, side, chunk)
  const int s = (int)(local % nchunk);
  const int pb = (int)((local / nchunk) % npb);
  const long long rest = local / nchunk / npb;
  const int p = pb * 256 + threadIdx.x;
  const int b = b0 + (int)(rest % B);
  const int side = (int)(rest / B) + side0;                  // 0 = src (k), 1 = tgt (q); side0 = 1: tgt only
  const int C = L.C, HW = L.HW, P = L.P, Ppad = L.Ppad, Cp8 = L.Cp >> 3;
  if (p >= Ppad) return;
  const bool valid = p < P;
  const int id = valid ? (keys_s != nullptr ? (int)(keys_s[p] >> 32) : __ldg(L.sid + p)) : 0;   // clamped to [0, HW) by the id prep
  const T* col = reinterpret_cast<const T*>(side ? L.tgt : L.src) + (size_t)b * C * HW + id;
  float v[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int c = s * 32 + k;
    v[k] = (valid && c < C) ? to_f32<T>(__ldcg(col + (size_t)c * HW)) : 0.f;
  }
  float ss = 0.f;
  bool bad = false;
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    ss = fmaf(v[k], v[k], ss);
    bad |= !isfinite(v[k]);
  }
  float* ssbase = side ? L.qss : L.kss;                      // NULL in head mode (the head's output is normalised)
  if (ssbase != nullptr) ssbase[((size_t)b * nchunk + s) * Ppad + p] = bad ? __int_as_float(0x7fc00000) : ss;
  __nv_bfloat16* hi_base = side ? L.qhi : L.khi;
  __nv_bfloat16* lo_base = side ? L.qlo : L.klo;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int c8 = s * 4 + g;
    size_t cm;                                                // core-matrix index
    if (side || L.head_src_rows) cm = (((size_t)b * (Ppad >> 7) + (p >> 7)) * Cp8 + c8) * 16 + ((p & 127) >> 3);
    else {                                                    // key blocks of <= 256 rows, one after the other
      const int nb8 = min(256, Ppad - pb * 256) >> 3;
      cm = (((size_t)b * Ppad + (size_t)pb * 256) * Cp8) / 8 + (size_t)c8 * nb8 + ((p & 255) >> 3);
    }
    const size_t off = cm * 64 + (size_t)(p & 7) * 8;         // elements
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float a = v[g * 8 + 2 * k], c2 = v[g * 8 + 2 * k + 1];
      const __nv_bfloat16 ah = __float2bfloat16_rn(a), ch = __float2bfloat16_rn(c2);
      const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah));
      const __nv_bfloat16 cl = __float2bfloat16_rn(c2 - __bfloat162float(ch));
      hw[k] = pack_bf16x2(ah, ch);
      lw[k] = pack_bf16x2(al, cl);
    }
    *reinterpret_cast<uint4*>(hi_base + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (lo_base != nullptr) *reinterpret_cast<uint4*>(lo_base + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    if (!side && !L.head_src_rows) {
      // second, key-major copy of K: [image][p/8][c/8][8 keys][8 ch] -- a chunk of 32 keys x all
      // channels is one contiguous bulk copy and is read MN-major (N = channel) by dQ = dZ K
      const size_t off2 = (((size_t)b * (Ppad >> 3) + (p >> 3)) * Cp8 + c8) * 64 + (size_t)(p & 7) * 8;
      *reinterpret_cast<uint4*>(L.k2hi + off2) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      if (L.k2lo != nullptr) *reinterpret_cast<uint4*>(L.k2lo + off2) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}

// grid = sum_l 2 * B * ceil(Ppad_l / 256) * nchunk_l
__global__ void __launch_bounds__(kThreads) k_gather_tc(const __grid_constant__ Params p,
                                                        const __grid_constant__ BlockMap m) {
  pdl_enter();
  const long long blk = blockIdx.x;
  if (blk == 0 && threadIdx.x == 0 && p.b0 == 0 && p.counter != nullptr) {
    // launch-sequence state of the loss kernel that follows on this stream (k_prep does the same when it
    // runs on this stream; with pnce_plan_ids it ran elsewhere, before the workspace existed)
    p.counter[0] = 0u; p.counter[1] = 0u;
    if (p.nonfinite != nullptr) p.nonfinite[1] = 0;
  }
  const int slot = find_layer(m, blk, p.n_layers);
  const int l = m.layer[slot];                                 // launch_gather_tc orders light layers first
  const long long local = blk - m.start[slot];
  if (p.dtype == PNCE_F32) gather_tc_chunk<float>(p.L[l], p.b0, p.bn, local, p.side0);
  else if (p.dtype == PNCE_F16) gather_tc_chunk<__half>(p.L[l], p.b0, p.bn, local, p.side0);
  else gather_tc_chunk<__nv_bfloat16>(p.L[l], p.b0, p.bn, local, p.side0);
}

// Small problems (launch_gather_tc: at most kFoldMaxCtas gather CTAs, ids not planned ahead): the id prep of k_prep is
// FOLDED into the gather -- every CTA draws (or reads) and sorts its layer's ids in shared memory (P <= 1024 keys, 36-55
// barrier steps: ~1.5 us beside its 32 sector loads per thread) and the first CTA of each layer also writes the tables the
// loss and dense kernels read (sid, perm, rank, cslot; the ids themselves in draw mode).  One launch and its 8-10 us on the
// critical path less per step: at B = 1 a step is four kernels of 10-25 us each.  Same values bit for bit: prep_layer is
// the one routine.  dynamic smem = N2max * 8 + 64.
constexpr int kFoldMaxCtas = 512;        // measured: B = 8 (384 CTAs) 149 -> 143 us per step, B = 16 (768 CTAs) 240 -> 242 us
__global__ void __launch_bounds__(kThreads) k_gather_tc_fold(const __grid_constant__ Params p,
                                                             const __grid_constant__ BlockMap m) {
  pdl_enter();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const long long blk = blockIdx.x;
  if (blk == 0 && threadIdx.x == 0 && p.b0 == 0 && p.counter != nullptr) {
    p.counter[0] = 0u; p.counter[1] = 0u;
    if (p.nonfinite != nullptr) p.nonfinite[1] = 0;
  }
  const int slot = find_layer(m, blk, p.n_layers);
  const int l = m.layer[slot];
  const long long local = blk - m.start[slot];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  prep_layer(p.L[l], keys, p.rng_draw, p.rng_seed, p.rng_offset + 4ull * (unsigned long long)l, local == 0);
  __syncthreads();
  if (p.dtype == PNCE_F32) gather_tc_chunk<float>(p.L[l], p.b0, p.bn, local, p.side0, keys);
  else if (p.dtype == PNCE_F16) gather_tc_chunk<__half>(p.L[l], p.b0, p.bn, local, p.side0, keys);
  else gather_tc_chunk<__nv_bfloat16>(p.L[l], p.b0, p.bn, local, p.side0, keys);
}

// Global negatives (pnce_mb_shard_keys), after the gather: flags[l] = 1 when a query row of layer l of this rank is
// non-finite -- the gather marks such a row's partial sums of squares with NaN (the padding rows hold 0).  The flags
// travel in the rank's slot next to its keys, so that every rank's finalize guards the layer on the rows of every rank.
// The caller zeroes the flags first; CTA (x, l) scans kMbQbadFloats of layer l's qss.  A separate launch rather than a
// store in the three gather variants: those are HBM-bound and shared by every mode, this reads ~1 % of their bytes
// back from L2.
constexpr int kMbQbadFloats = kThreads * 16;
__global__ void __launch_bounds__(kThreads) k_mb_qbad(const __grid_constant__ Params p, int* flags) {
  pdl_enter();
  const int l = blockIdx.y;
  const LayerDev& L = p.L[l];
  const size_t n4 = (size_t)p.B * L.nchunk * L.Ppad / 4;     // Ppad is a multiple of 128
  const float4* q = reinterpret_cast<const float4*>(L.qss);
  bool bad = false;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const size_t i = (size_t)blockIdx.x * (kMbQbadFloats / 4) + k * kThreads + threadIdx.x;
    if (i < n4) {
      const float4 v = __ldcg(q + i);
      bad |= !(v.x == v.x) || !(v.y == v.y) || !(v.z == v.z) || !(v.w == v.w);
    }
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) flags[l] = 1;
}

// netF head with minibatch negatives (pnce_head_mb_fwd), after the head's second GEMM: the group guard needs a sampled
// patch holding a NaN / Inf to make its layer non-finite, but the head's ReLU (fmaxf) turns a NaN row of X W1^T into
// zeros, so the head's output would be finite.  The gather marks such a raw row in xqss / xkss (NaN partial sums of
// squares); this kernel carries the mark onto the head output's sums of squares (chunk 0 of yqss / ykss), where the
// loss kernel reads it as a non-finite row or key and guards the layer.  A marked query row of X is also zeroed: the
// guarded layer's dY is zero, and dW1 = dH^T X must then be 0, not 0 * NaN.  One thread per (layer, image, slot).
struct HeadGuardLayer {
  const float* xqss;           // [B][nchunk][Ppad] of the raw patches (the gather's marks)
  const float* xkss;
  float* yqss;                 // [B][ncy][Ppad] of the head's output
  float* ykss;
  __nv_bfloat16* xq_hi;        // raw query rows: the row blob the gather writes (tile-major, 8-channel core matrices)
  __nv_bfloat16* xq_lo;        // NULL in single-pass bf16
  int P, Ppad, Cp8, nchunk, ncy;
};
struct HeadGuardLaunch {
  HeadGuardLayer L[PNCE_MAX_LAYERS];
  int B;
};

__global__ void __launch_bounds__(kThreads) k_head_mb_guard(const __grid_constant__ HeadGuardLaunch g) {
  pdl_enter();
  const HeadGuardLayer& L = g.L[blockIdx.y];
  const long long r = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (r >= (long long)g.B * L.Ppad) return;
  const int b = (int)(r / L.Ppad), p = (int)(r % L.Ppad);
  if (p >= L.P) return;
  bool bq = false, bk = false;
  for (int s = 0; s < L.nchunk; ++s) {
    const size_t i = ((size_t)b * L.nchunk + s) * L.Ppad + p;
    const float q = __ldcg(L.xqss + i), k = __ldcg(L.xkss + i);
    bq |= !(q == q);
    bk |= !(k == k);
  }
  const float nan = __int_as_float(0x7fc00000);
  if (bk) L.ykss[(size_t)b * L.ncy * L.Ppad + p] = nan;
  if (bq) {
    L.yqss[(size_t)b * L.ncy * L.Ppad + p] = nan;
    for (int c8 = 0; c8 < L.Cp8; ++c8) {
      const size_t cm = (((size_t)b * (L.Ppad >> 7) + (p >> 7)) * L.Cp8 + c8) * 16 + ((p & 127) >> 3);
      const size_t off = cm * 64 + (size_t)(p & 7) * 8;
      *reinterpret_cast<uint4*>(L.xq_hi + off) = make_uint4(0u, 0u, 0u, 0u);
      if (L.xq_lo != nullptr) *reinterpret_cast<uint4*>(L.xq_lo + off) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
}

// One CTA per layer: ids -> (sid, perm, rank, ustart, bitmap, prefix); CTA 0 also resets the
// last-CTA counter and the protocol flag of the launch sequence.
__global__ void __launch_bounds__(kThreads) k_prep(const __grid_constant__ Params p) {
  pdl_enter();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int l = blockIdx.x;
  if (l == 0 && threadIdx.x == 0 && p.counter != nullptr) {
    p.counter[0] = 0u; p.counter[1] = 0u;
    if (p.nonfinite != nullptr) p.nonfinite[1] = 0;
  }
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  int N2 = 1;
  while (N2 < p.L[l].P) N2 <<= 1;
  prep_layer(p.L[l], keys, p.rng_draw, p.rng_seed, p.rng_offset + 4ull * (unsigned long long)l);
}

}  // namespace pnce
