// Tensor-core path, launch 3: fused logits + diagonal CE forward/backward on tcgen05.
// One CTA per (layer, image, 128-row half of the P x P logits); 192 threads, warp-specialised:
//   warp 0      bulk-copy producer (TMA engine, 1-D, operand blobs are pre-tiled by k_gather_tc)
//   warp 1      TMEM owner + the single MMA-issuing thread
//   warps 2..5  epilogue: one thread per logits row (TMEM lane), tcgen05.ld -> registers
// Rows are in SORTED-ID order (k_gather_tc gathers slot i = i-th smallest id): the loss is invariant
// under a common permutation of q and k rows, and the gradient rows then leave as coalesced stores
// in exactly the order the dense backward reads them.
//
//   phase 1   Z(128 x N) = Q_half K^T           kind::f16 bf16, fp32 accumulate in TMEM cols [0,N)
//             streamed over C in chunks of 32 channels through a 4-slot ring (2 slots live in the dZ
//             region, idle until the epilogue), so the bulk copies run 3 stages ahead of the MMAs.
//             bf16x3 mode issues hi*hi + hi*lo + lo*hi into the same accumulator (~2^-17 operand error).
//   epilogue  y_ij = acc * (log2e/tau)(1/||q_i||)(1/||k_j||)   (logits in log2 units), clamp, row sum of
//             exp2, diagonal pick, row loss (warp-shuffle reduced), dZ = (softmax - I) * mask / (P B L),
//             s_i = sum_j dZ_ij z_ij (= q_hat . dq, no second reduction needed),
//             dZ_ij / ||k_j|| split hi/lo -> shared memory as the next MMA's A operand.
//             The element loops are branch-free (32 independent columns per tcgen05.ld).
//   phase 2   dQ(128 x C) = dZ K               K streamed a second time, KEY-major (32 keys x all channels
//             per 3-slot ring stage, from the gather's second K blob) and read MN-major, so every MMA
//             is M128 x N=C x K16 (N=32 MMAs re-read the whole A tile and starve on shared-memory
//             bandwidth).  Chunk j's MMAs start as soon as the four epilogue warps have written
//             dZ[:, 32j..32j+31]: phase 2 overlaps pass B.  Accumulator: TMEM cols [256, 256+C)
//   epilogue  dq/tau, normalise backward (raw q re-read from the Q operand blob, hi + lo),
//             dxT[b][c][slot] (unit upstream gradient), coalesced.
// The logits, softmax and dZ never leave the SM.  Replaces patchnce_cut.py:83-110 and the autograd
// backward of :77-94 (SURVEY.md section 8 rows a7-a11).  Shapes: P <= 1024, C <= 256.
// P > 256: the keys are processed in blocks of 256 (flash-style): pass 1 accumulates the row sums block
// by block, pass 2 recomputes each logits block, turns it into dZ and accumulates dQ += dZ_blk K_blk.
#pragma once
#include "common.cuh"
#include "loss_simt.cuh"
#include "umma.cuh"

namespace pnce {

constexpr int kTcThreads = 192;
constexpr int kTcStageBytes = 49152;        // Qhi 8K | Qlo 8K | Khi 16K | Klo 16K   (32 channels)
constexpr int kTcOffQlo = 8192, kTcOffKhi = 16384, kTcOffKlo = 32768;
constexpr int kTcDzBytes = 65536;           // 128 x 256 bf16
constexpr int kTcSmemBytes = 2 * kTcStageBytes + 2 * kTcDzBytes + 1024 /*invk*/ + 256 /*barriers, misc*/;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

constexpr int kTcSlots1 = 4;                // phase-1 slots: 2 in the ring region + 2 in the (still idle) dZ region
constexpr int kTcSlots2 = 3;                // phase-2 slots (K only, 32 KB each) in the ring region
constexpr int kTcStage2Bytes = 32768;       // Khi 16K | Klo 16K

struct TcShared {
  uint64_t full1[kTcSlots1], empty1[kTcSlots1], full2[kTcSlots2], empty2[kTcSlots2], zfull, dzready[8], dqfull, zfree, p2done;
  uint32_t tmem_base;
  int dead;
  int flag;
  int badk;                                  // some key row of this image is non-finite
  float red[4];
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t bf16x2_bits(float lo_elem, float hi_elem) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo_elem, hi_elem);   // .x = first (low 16 bits)
  return *reinterpret_cast<const uint32_t*>(&v);
}

// ---- pass A over one 32-column chunk: sum of exp2 of the (clamped) logits, 4 partial sums -------
// CLAMP: the +-50 clamp can bind (1/tau > 50).  Padding columns carry w = 0 -> y = 0 -> exp2 = 1
// exactly; the caller subtracts their count.
template <bool CLAMP>
__device__ __forceinline__ void tc_pass_a(const uint32_t (&r)[32], const float* __restrict__ wk, float a,
                                          float cl, float (&se)[4]) {
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) {
    const float4 w = *reinterpret_cast<const float4*>(wk + k4 * 4);
    const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float y = __uint_as_float(r[k4 * 4 + t]) * a * ww[t];
      if (CLAMP) y = fminf(fmaxf(y, -cl), cl);
      se[t] += ex2f(y);
    }
  }
}

// The same for the LAST chunk of a key block when it holds padding columns (key weight w == 0): those
// columns are excluded by a select instead of being counted as exp2(0) = 1 and subtracted afterwards -- the
// subtraction cancels catastrophically when every real logit of the row is very negative (sum of exp2 below
// one ulp of the pad count: P = 1, C = 1, constant maps ...), found by scratch/stress.py.  A key with w == 0
// that is NOT padding is a non-finite row, and the image is guarded anyway.
template <bool CLAMP>
__device__ __forceinline__ void tc_pass_a_masked(const uint32_t (&r)[32], const float* __restrict__ wk, float a,
                                                 float cl, float (&se)[4]) {
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) {
    const float4 w = *reinterpret_cast<const float4*>(wk + k4 * 4);
    const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float y = __uint_as_float(r[k4 * 4 + t]) * a * ww[t];
      if (CLAMP) y = fminf(fmaxf(y, -cl), cl);
      se[t] += (ww[t] != 0.f) ? ex2f(y) : 0.f;
    }
  }
}

// ---- pass B over one 32-column chunk: softmax * coef / ||k_j|| -> bf16 hi (+lo) A-operand rows,
//      s2 += dZ * y.  The "- I" of the diagonal is patched in afterwards by the owning thread.
//      Padding columns: w = 0 -> the stored operand and the s2 term are exactly 0.
template <bool CLAMP>
__device__ __forceinline__ void tc_pass_b(const uint32_t (&r)[32], const float* __restrict__ wk, float a,
                                          float cl, float lse2, float coef, bool x3, unsigned char* dzhi,
                                          unsigned char* dzlo, uint32_t off0, float& s2) {
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    float dd[8];
#pragma unroll
    for (int h4 = 0; h4 < 2; ++h4) {
      const float4 w = *reinterpret_cast<const float4*>(wk + g8 * 8 + h4 * 4);
      const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float y = __uint_as_float(r[g8 * 8 + h4 * 4 + t]) * a * ww[t];
        const float yc = CLAMP ? fminf(fmaxf(y, -cl), cl) : y;
        float d = ex2f(yc - lse2) * coef;
        if (CLAMP) d = (fabsf(y) <= cl) ? d : 0.f;             // clamp backward mask (inclusive)
        s2 = fmaf(d, y, s2);
        dd[h4 * 4 + t] = d * ww[t];
      }
    }
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int k2 = 0; k2 < 4; ++k2) {
      hw[k2] = bf16x2_bits(dd[2 * k2], dd[2 * k2 + 1]);
      const float r0 = dd[2 * k2] - __uint_as_float(hw[k2] << 16);
      const float r1 = dd[2 * k2 + 1] - __uint_as_float(hw[k2] & 0xffff0000u);
      lw[k2] = bf16x2_bits(r0, r1);
    }
    const uint32_t off = off0 + (uint32_t)g8 * 2048u;          // next 8-column slab of the A operand
    *reinterpret_cast<uint4*>(dzhi + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (x3) *reinterpret_cast<uint4*>(dzlo + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}

// ---- single-pass softmax over one 32-column chunk (key-blocked kernel, P > 256, clamp cannot bind): e = exp2(y) once,
//      the UNNORMALISED e / ||k_j|| is the dQ operand, se += e (padding columns masked), s2 += e y.  The row factor
//      coef / se and the "- I" term are applied afterwards (the diagonal entry is patched once se is complete).
__device__ __forceinline__ void tc_pass_single(const uint32_t (&r)[32], const float* __restrict__ wk, float a, bool x3,
                                               unsigned char* dzhi, unsigned char* dzlo, uint32_t off0, float (&se)[4],
                                               float& s2) {
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    float dd[8];
#pragma unroll
    for (int h4 = 0; h4 < 2; ++h4) {
      const float4 w = *reinterpret_cast<const float4*>(wk + g8 * 8 + h4 * 4);
      const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float y = __uint_as_float(r[g8 * 8 + h4 * 4 + t]) * a * ww[t];
        const float e = ex2f(y);
        se[t] += (ww[t] != 0.f) ? e : 0.f;
        s2 = fmaf(e, y, s2);
        dd[h4 * 4 + t] = e * ww[t];
      }
    }
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int k2 = 0; k2 < 4; ++k2) {
      hw[k2] = bf16x2_bits(dd[2 * k2], dd[2 * k2 + 1]);
      const float r0 = dd[2 * k2] - __uint_as_float(hw[k2] << 16);
      const float r1 = dd[2 * k2 + 1] - __uint_as_float(hw[k2] & 0xffff0000u);
      lw[k2] = bf16x2_bits(r0, r1);
    }
    const uint32_t off = off0 + (uint32_t)g8 * 2048u;
    *reinterpret_cast<uint4*>(dzhi + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (x3) *reinterpret_cast<uint4*>(dzlo + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}
// Key-block and chunk order of an item in single-pass mode: the block that holds the diagonals of the item's own 128 rows
// goes LAST, and inside it the (up to) four chunks with those diagonals go last -- they are released only when the row
// sums are complete.  dlo = first diagonal chunk of that block (0 or 4), nch = its chunks that hold real columns.
__device__ __forceinline__ int tc_block_at(int o, int nkb, int kbd) { return o < nkb - 1 ? (o < kbd ? o : o + 1) : kbd; }
__device__ __forceinline__ int tc_chunk_last(int k, int nch, int dlo) {
  const int nn = dlo == 0 ? (nch > 4 ? nch - 4 : 0) : (nch < 4 ? nch : 4);      // chunks without diagonals come first
  return k < nn ? (dlo == 0 ? k + 4 : k) : dlo + (k - nn);
}

// Both passes walk the row in 32-column chunks with two STATIC register buffers so that the
// tcgen05.ld of chunk ch+1 is in flight while chunk ch is processed.
template <bool CLAMP>
__device__ __forceinline__ void tc_row_pass_a(uint32_t trow, int nch, const float* __restrict__ invk_s, float a,
                                              float cl, int chd, int lane, float (&se)[4], float& ydraw, bool pad) {
  using namespace umma;
  uint32_t r0[32], r1[32];
  tmem_ld32(trow, r0);
  for (int ch = 0; ch < nch; ch += 2) {
    tmem_ld_wait();
    if (ch + 1 < nch) tmem_ld32(trow + (ch + 1) * 32, r1);
    if (pad && ch == nch - 1) tc_pass_a_masked<CLAMP>(r0, invk_s + ch * 32, a, cl, se);
    else tc_pass_a<CLAMP>(r0, invk_s + ch * 32, a, cl, se);
    if (ch == chd) {
#pragma unroll
      for (int k = 0; k < 32; ++k) ydraw = (k == lane) ? __uint_as_float(r0[k]) : ydraw;
    }
    if (ch + 1 < nch) {
      tmem_ld_wait();
      if (ch + 2 < nch) tmem_ld32(trow + (ch + 2) * 32, r0);
      if (pad && ch + 1 == nch - 1) tc_pass_a_masked<CLAMP>(r1, invk_s + (ch + 1) * 32, a, cl, se);
      else tc_pass_a<CLAMP>(r1, invk_s + (ch + 1) * 32, a, cl, se);
      if (ch + 1 == chd) {
#pragma unroll
        for (int k = 0; k < 32; ++k) ydraw = (k == lane) ? __uint_as_float(r1[k]) : ydraw;
      }
    }
  }
}

// the "- I" of (softmax - I): the thread that owns row i rewrites its diagonal element
struct TcDiag {
  bool rowok, pass;
  float d_w;                 // (p_ii - 1) * coef / ||k_i||, or 0 when the clamp masks it
  uint32_t off;              // byte offset of the element in the dZ operand
};
__device__ __forceinline__ void tc_fix_diag(const TcDiag& dg, bool x3, unsigned char* dzhi, unsigned char* dzlo) {
  if (dg.rowok) {
    const __nv_bfloat16 hi = __float2bfloat16_rn(dg.d_w);
    *reinterpret_cast<__nv_bfloat16*>(dzhi + dg.off) = hi;
    if (x3) *reinterpret_cast<__nv_bfloat16*>(dzlo + dg.off) = __float2bfloat16_rn(dg.d_w - __bfloat162float(hi));
  }
}

template <bool CLAMP>
__device__ __forceinline__ void tc_row_pass_b(uint32_t trow, int nch, const float* __restrict__ invk_s, float a,
                                              float cl, float lse2, float coef, bool x3, unsigned char* dzhi,
                                              unsigned char* dzlo, uint32_t rowoff, int chd, const TcDiag& dg,
                                              uint64_t* dzready, float& s2) {
  using namespace umma;
  uint32_t r0[32], r1[32];
  tmem_ld32(trow, r0);
  for (int ch = 0; ch < nch; ch += 2) {
    tmem_ld_wait();
    if (ch + 1 < nch) tmem_ld32(trow + (ch + 1) * 32, r1);
    tc_pass_b<CLAMP>(r0, invk_s + ch * 32, a, cl, lse2, coef, x3, dzhi, dzlo, (uint32_t)(ch * 4) * 2048u + rowoff, s2);
    if (ch == chd) tc_fix_diag(dg, x3, dzhi, dzlo);
    fence_proxy_async_smem();
    mbar_arrive(&dzready[ch]);                               // 128 arrivals release chunk ch to the MMA thread
    if (ch + 1 < nch) {
      tmem_ld_wait();
      if (ch + 2 < nch) tmem_ld32(trow + (ch + 2) * 32, r0);
      tc_pass_b<CLAMP>(r1, invk_s + (ch + 1) * 32, a, cl, lse2, coef, x3, dzhi, dzlo,
                       (uint32_t)((ch + 1) * 4) * 2048u + rowoff, s2);
      if (ch + 1 == chd) tc_fix_diag(dg, x3, dzhi, dzlo);
      fence_proxy_async_smem();
      mbar_arrive(&dzready[ch + 1]);
    }
  }
}

// Raw q values of one 32-channel chunk of this thread's row, re-read from the Q operand blob (hi + lo
// = the fp32 value to 2^-17; the blob was streamed through this SM a few microseconds ago, so these are
// L2 hits): 4 slabs x (16 B hi + 16 B lo).
struct TcQChunk {
  uint4 h[4], l[4];
};
__device__ __forceinline__ void tc_q_load(TcQChunk& qc, const __nv_bfloat16* __restrict__ qh,
                                          const __nv_bfloat16* __restrict__ ql, int s, int nstage) {
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    const bool in = s < nstage;
    qc.h[g8] = in ? __ldcg(reinterpret_cast<const uint4*>(qh + (size_t)(s * 4 + g8) * 1024)) : make_uint4(0u, 0u, 0u, 0u);
    qc.l[g8] = (in && ql != nullptr) ? __ldcg(reinterpret_cast<const uint4*>(ql + (size_t)(s * 4 + g8) * 1024))
                                     : make_uint4(0u, 0u, 0u, 0u);
  }
}
__device__ __forceinline__ void tc_q_unpack(const TcQChunk& qc, float (&q)[32]) {
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    const uint32_t hw[4] = {qc.h[g8].x, qc.h[g8].y, qc.h[g8].z, qc.h[g8].w};
    const uint32_t lw[4] = {qc.l[g8].x, qc.l[g8].y, qc.l[g8].z, qc.l[g8].w};
#pragma unroll
    for (int k2 = 0; k2 < 4; ++k2) {
      q[g8 * 8 + 2 * k2] = __uint_as_float(hw[k2] << 16) + __uint_as_float(lw[k2] << 16);
      q[g8 * 8 + 2 * k2 + 1] = __uint_as_float(hw[k2] & 0xffff0000u) + __uint_as_float(lw[k2] & 0xffff0000u);
    }
  }
}

// dxT stores carry an L2 evict_last policy: the rows (50 MB at B=64) are then still in L2 when the dense
// backward reads them, instead of having been pushed out by the blob traffic of the rest of this kernel --
// reads that would interleave with the dense kernel's 7 TB/s write stream (measured: dense 464 -> 454 us,
// step 896 -> 877 us; pnce_debug_set key 9 = 0 turns it off).  k_dense_flat reads them with ld.global.cs,
// which hands the lines back to the replacement policy as soon as they are consumed.
#ifdef PNCE_EXPERIMENTS
__device__ int g_dx_evict_last = 1;
#else
constexpr int g_dx_evict_last = 1;
#endif
__device__ __forceinline__ void st_dx(float* p, float v, bool keep, uint64_t pol) {
  if (keep) asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
  else *p = v;
}
__device__ __forceinline__ void st_dx4(float* p, float a, float b, float c, float d, bool keep, uint64_t pol) {
  if (keep)
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "l"(pol)
                 : "memory");
  else *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
// one whole 32-byte sector per lane (sm_100: STG.256); 128-bit row stores from 32 different rows are 32 HALF sectors
__device__ __forceinline__ void st_dx8(float* p, const float* v, bool keep, uint64_t pol) {
  if (keep)
    asm volatile("st.global.L2::cache_hint.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8}, %9;" ::"l"(p), "f"(v[0]), "f"(v[1]),
                 "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "l"(pol)
                 : "memory");
  else
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// dQ epilogue for one 32-channel chunk; NPC = pitch of dxT rows (compile-time: immediates; 0 = run time).
// Head mode (dyh != NULL): the gradient w.r.t. the head output leaves as a bf16 hi(+lo) row blob
// (the A operand of the head's backward GEMMs) instead of fp32 rows; padding rows are written as 0.
// rm (channels-last maps, nhwc.cuh): the rows leave ROW-major -- dp = this row's 32 channels, np_rt = C; every
// thread writes one whole 128-byte line.
template <int NPC>
__device__ __forceinline__ void tc_dq_chunk(const uint32_t (&r)[32], const TcQChunk& qc, float* __restrict__ dp,
                                            int nvalid, float c1, float c2, bool rowok, __nv_bfloat16* dyh,
                                            __nv_bfloat16* dyl, int np_rt, bool rm = false) {
  const size_t NP = NPC ? (size_t)NPC : (size_t)np_rt;
  float qv[32], out[32];
  tc_q_unpack(qc, qv);
#pragma unroll
  for (int k = 0; k < 32; ++k) out[k] = fmaf(-qv[k], c2, __uint_as_float(r[k]) * c1);
  if (dyh != nullptr) {
#pragma unroll
    for (int g8 = 0; g8 < 4; ++g8) {
      uint32_t h[4], l[4];
#pragma unroll
      for (int k2 = 0; k2 < 4; ++k2) {
        const float a0 = rowok ? out[g8 * 8 + 2 * k2] : 0.f, a1 = rowok ? out[g8 * 8 + 2 * k2 + 1] : 0.f;
        h[k2] = bf16x2_bits(a0, a1);
        l[k2] = bf16x2_bits(a0 - __uint_as_float(h[k2] << 16), a1 - __uint_as_float(h[k2] & 0xffff0000u));
      }
      *reinterpret_cast<uint4*>(dyh + g8 * 1024) = make_uint4(h[0], h[1], h[2], h[3]);
      if (dyl != nullptr) *reinterpret_cast<uint4*>(dyl + g8 * 1024) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    return;
  }
  if (rowok && g_dx_evict_last != 2) {                         // 2: experiment knob (no stores at all)
    const bool keep = g_dx_evict_last != 0;
    uint64_t pol = 0;
    if (keep) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    if (rm) {
      if (nvalid >= 32 && (np_rt & 7) == 0) {
#pragma unroll
        for (int k8 = 0; k8 < 4; ++k8) st_dx8(dp + k8 * 8, out + k8 * 8, keep, pol);
      } else if (nvalid >= 32 && (np_rt & 3) == 0) {
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) st_dx4(dp + k4 * 4, out[k4 * 4], out[k4 * 4 + 1], out[k4 * 4 + 2], out[k4 * 4 + 3], keep, pol);
      } else {
#pragma unroll
        for (int k = 0; k < 32; ++k)
          if (k < nvalid) st_dx(dp + k, out[k], keep, pol);
      }
      return;
    }
    if (nvalid >= 32) {
#pragma unroll
      for (int k = 0; k < 32; ++k) st_dx(dp + k * NP, out[k], keep, pol);
    } else {
#pragma unroll
      for (int k = 0; k < 32; ++k)
        if (k < nvalid) st_dx(dp + k * NP, out[k], keep, pol);
    }
  }
}

template <int NPC>
__device__ __forceinline__ void tc_dq_epilogue(uint32_t tacc, int nstage, int C, const __nv_bfloat16* __restrict__ qh,
                                               const __nv_bfloat16* __restrict__ ql, float* __restrict__ dxrow,
                                               float c1, float c2, bool rowok, __nv_bfloat16* dyh,
                                               __nv_bfloat16* dyl, uint64_t* dqfull, volatile int* dead,
                                               TcQChunk& qa, TcQChunk& qb, int np_rt = 0, uint32_t parity = 0u,
                                               bool rm = false) {
  using namespace umma;
  const size_t NP = rm ? (size_t)1 : (NPC ? (size_t)NPC : (size_t)np_rt);   // rm: dxrow is this row, channels contiguous
  mbar_wait(dqfull, parity, dead);
  tc_fence_after();
  for (int s = 0; s < nstage; s += 2) {
    uint32_t r[32];
    tmem_ld32(tacc + s * 32, r);
    tmem_ld_wait();
    tc_dq_chunk<NPC>(r, qa, dxrow + (size_t)s * 32 * NP, C - s * 32, c1, c2, rowok,
                     dyh ? dyh + (size_t)s * 4096 : nullptr, dyl ? dyl + (size_t)s * 4096 : nullptr, np_rt, rm);
    tc_q_load(qa, qh, ql, s + 2, nstage);                     // two chunks ahead (static double buffer)
    if (s + 1 < nstage) {
      tmem_ld32(tacc + (s + 1) * 32, r);
      tmem_ld_wait();
      tc_dq_chunk<NPC>(r, qb, dxrow + (size_t)(s + 1) * 32 * NP, C - (s + 1) * 32, c1, c2, rowok,
                       dyh ? dyh + (size_t)(s + 1) * 4096 : nullptr, dyl ? dyl + (size_t)(s + 1) * 4096 : nullptr,
                       np_rt, rm);
      tc_q_load(qb, qh, ql, s + 3, nstage);
    }
  }
}

// Global negatives: where key image bk (a global image index) lives -- slot bk / B of p.kslot bytes, image bk % B inside
// it.  GN = false (one rank): the caller's own blobs, image bk.
template <bool GN>
__device__ __forceinline__ size_t tc_mb_key_slot(const Params& p, int bk, int& local) {
  if (!GN) {
    local = bk;
    return 0;
  }
  const int w = bk / p.B;
  local = bk - w * p.B;
  return (size_t)w * p.kslot;
}

// 1/||k_j|| of the 256 keys [key0, key0 + 256) of image bk, folded from the gather's partial sums of squares (minibatch
// mode: an item walks the keys of every image, so the weights are built per key block instead of once per image; 8 KB
// of L2 reads per block next to the 64-256 KB of operand bytes the block streams).  A non-finite key raises badk.
template <bool GN>
__device__ __forceinline__ float tc_mb_key_weight(const Params& p, const LayerDev& L, int bk, int key, int nstage) {
  int lb;
  const float* kss = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(L.kss) + tc_mb_key_slot<GN>(p, bk, lb));
  float ss = 0.f;
  for (int s = 0; s < nstage; ++s) ss += __ldcg(kss + ((size_t)lb * nstage + s) * L.Ppad + key);
  const float nrm = sqrtf(ss);
  return (nrm == nrm) ? 1.0f / fmaxf(nrm, kNormEps) : nrm;      // NaN: the gather saw a non-finite element
}
template <bool GN>
__device__ __forceinline__ void tc_mb_key_weights(const Params& p, const LayerDev& L, int bk, int key0, int nstage, int et,
                                                  float* invk_s, int* badk) {
  asm volatile("bar.sync 1, 128;" ::: "memory");
  for (int j = et; j < 256; j += 128) {
    const int key = key0 + j;
    float w = 0.f;
    if (key < L.P) {
      w = tc_mb_key_weight<GN>(p, L, bk, key, nstage);
      if (!(w == w)) { *badk = 1; w = 0.f; }
    }
    invk_s[j] = w;
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
}

// MB = false: k_loss_tc, one image's P x P problem per item.  MB = true: k_loss_tc_mb (minibatch negatives): the item
// (layer, image b, 128-row half) walks the key blocks (b', kb) of EVERY image of the batch -- the K blobs of the batch
// are one key-blocked blob of B * Ppad keys, and the ids are shared, so the sorted-slot order is a common permutation of
// all rows.  The item's own block (b, kb(row)) goes last, its diagonal chunks last.  GN = true (MB only):
// k_loss_tc_mb_gn, global negatives -- the key images are those of every rank's slot (tc_mb_key_slot) and the item's
// image is global image kimg0 + b, so a rank walks exactly the blocks, in exactly the order, that one GPU walks for the
// same row (a template parameter: as runtime fields the slot arithmetic cost k_loss_tc_mb ~1 % at B = 16 and 64).
// Rows mode (p.rows_mode, MB only): rows are used as given and d loss / d q leaves row-major in dq_rows.
template <bool MB, bool GN = false>
__device__ __forceinline__ void loss_tc_body(const Params& p, const BlockMap& m) {
  extern __shared__ __align__(1024) unsigned char smem[];
  using namespace umma;
  unsigned char* stage0 = smem;
  unsigned char* dzhi = smem + 2 * kTcStageBytes;
  unsigned char* dzlo = dzhi + kTcDzBytes;
  float* invk_s = reinterpret_cast<float*>(dzlo + kTcDzBytes);
  TcShared* sh = reinterpret_cast<TcShared*>(invk_s + 256);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int slot_l = find_layer(m, blockIdx.x, p.n_layers);
  const int l = m.layer[slot_l];
  const LayerDev& L = p.L[l];
  const int local = (int)(blockIdx.x - m.start[slot_l]);
  const int halves = L.Ppad >> 7;
  const int mh = local % halves, b = p.b0 + local / halves;
  const int Ppad = L.Ppad, P = L.P, C = L.C, Cp = L.Cp, Cp8 = L.Cp >> 3, nstage = L.nchunk;
  // keys are processed in blocks of <= 256 (the logits block must fit 256 TMEM columns next to the dQ
  // accumulator).  One block (P <= 256): Z is computed once.  More blocks: flash-style two passes --
  // pass 1 accumulates the row sums of exp2 block by block, pass 2 recomputes each Z block for dZ.
  // minibatch mode: nkb counts the blocks of every image, block g = image g / nkbi, block g % nkbi of that image
  // global negatives: the key images are the kworld * B images of every rank's slot, this item's image is global
  // image gb = kimg0 + b (its diagonal block and diagonal key weight)
  const int nkbi = (Ppad + 255) >> 8;
  const int nkb = MB ? (GN ? p.kworld : 1) * p.B * nkbi : nkbi;
  const int gb = GN ? p.kimg0 + b : b;
  const bool multi = nkb > 1;
  const int nslots1 = multi ? 2 : kTcSlots1;                  // the dZ region is busy in pass 2 of the multi-block case
  const bool x3 = (p.math == PNCE_MATH_TC_BF16X3);
  // more than one key block and the +-50 clamp cannot bind (|cos| <= 1, every CUT temperature): ONE pass per block --
  // exp2 once, unnormalised operand, no recomputation of the logits (the two-pass form stays for clamp-binding tau).
  // Minibatch mode has no running maximum either: the row sum stays below N 2^(1.02 log2e / tau), finite in fp32 for
  // N = B * Ppad <= 65536 at every tau where the clamp cannot bind.
  const bool single = multi && !((1.0f / p.tau) * 1.02f > kClamp);
  const int kbd_item = (MB ? gb * nkbi : 0) + ((mh * 128) >> 8);   // key block with the diagonals of this item's rows
  const int dlo_item = ((mh * 128) & 255) >> 5;               // and the first of its (up to four) diagonal chunks
  volatile int* dead = &sh->dead;
  long long* tr = nullptr;                                   // debug stamps (pnce_debug_set key 3)
  if (p.trace != nullptr && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2)) tr = p.trace + (blockIdx.x ? 16 : 0);
#ifdef PNCE_EXPERIMENTS
#define PNCE_TR(slot) do { if (tr) tr[slot] = clock64(); } while (0)
#else
#define PNCE_TR(slot) do { } while (0)
#endif
  // debug timeline: (sm id, start ns, end ns) of every CTA at trace[64 + 3 * blockIdx.x]
  if (p.trace != nullptr && tid == 0) {
    unsigned sm; unsigned long long t;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.trace[64 + 3 * (size_t)blockIdx.x] = sm;
    p.trace[64 + 3 * (size_t)blockIdx.x + 1] = (long long)t;
  }

  if (tid == 0) {
    for (int k = 0; k < kTcSlots1; ++k) { mbar_init(&sh->full1[k], 1); mbar_init(&sh->empty1[k], 1); }
    for (int k = 0; k < kTcSlots2; ++k) { mbar_init(&sh->full2[k], 1); mbar_init(&sh->empty2[k], 1); }
    mbar_init(&sh->zfull, 1); mbar_init(&sh->dqfull, 1); mbar_init(&sh->zfree, 128); mbar_init(&sh->p2done, 1);
    for (int k = 0; k < 8; ++k) mbar_init(&sh->dzready[k], 128);
    sh->dead = 0;
    sh->badk = 0;
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(&sh->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                                                 // prologue done: now wait for the prerequisite grids
  const uint32_t tmem = sh->tmem_base;
  const int npass = (multi && !single) ? 2 : 1;

  if (warp == 0) {
    // ===================== producer =====================
    if (lane == 0) {
      const unsigned char* gq_hi = reinterpret_cast<const unsigned char*>(L.qhi) + ((size_t)b * halves + mh) * Cp8 * 2048;
      const unsigned char* gq_lo = reinterpret_cast<const unsigned char*>(L.qlo) + ((size_t)b * halves + mh) * Cp8 * 2048;
      const uint32_t k2bytes = (uint32_t)Cp * 64u;            // 32 keys x Cp channels x 2 B
      uint32_t it1 = 0, it2 = 0, nz = 0;
      bool ok = true;
      for (int pass = 0; pass < npass && ok; ++pass) {
        for (int o = 0; o < nkb && ok; ++o) {
          const int g = single ? tc_block_at(o, nkb, kbd_item) : o;
          const int kb = MB ? g % nkbi : g;                  // block of the keys, in image g / nkbi (minibatch mode)
          int lb = b;
          const size_t kslot = MB ? tc_mb_key_slot<GN>(p, g / nkbi, lb) : 0;
          const size_t kimg = kslot + (size_t)lb * Ppad * Cp * 2;
          const unsigned char* gk_hi = reinterpret_cast<const unsigned char*>(L.khi) + kimg;
          const unsigned char* gk_lo = reinterpret_cast<const unsigned char*>(L.klo) + kimg;
          const unsigned char* g2_hi = reinterpret_cast<const unsigned char*>(L.k2hi) + kimg;
          const unsigned char* g2_lo = reinterpret_cast<const unsigned char*>(L.k2lo) + kimg;
          const int NB = min(256, Ppad - kb * 256);           // keys of this block (128 or 256)
          const uint32_t kbytes = (uint32_t)NB * 64u;         // one K chunk: 4 slabs x NB/8 core matrices x 128 B
          const size_t kblk = (size_t)kb * 256 * Cp * 2;      // blocks are stored one after the other
          for (int s = 0; s < nstage && ok; ++s, ++it1) {     // Z block: Q and K chunks of 32 channels
            const int slot = it1 % nslots1;
            ok = mbar_wait(&sh->empty1[slot], ((it1 / nslots1) & 1u) ^ 1u, dead);
            if (!ok) break;
            unsigned char* st = stage0 + slot * kTcStageBytes;
            mbar_expect_tx(&sh->full1[slot], (8192u + kbytes) * (x3 ? 2u : 1u));
            bulk_g2s(st, gq_hi + (size_t)s * 8192, 8192u, &sh->full1[slot]);
            if (x3) bulk_g2s(st + kTcOffQlo, gq_lo + (size_t)s * 8192, 8192u, &sh->full1[slot]);
            bulk_g2s(st + kTcOffKhi, gk_hi + kblk + (size_t)s * kbytes, kbytes, &sh->full1[slot]);
            if (x3) bulk_g2s(st + kTcOffKlo, gk_lo + kblk + (size_t)s * kbytes, kbytes, &sh->full1[slot]);
          }
          // stay in lock-step with the MMA thread (a parity wait must never lag two phases behind)
          if (ok) ok = mbar_wait(&sh->zfull, nz & 1u, dead);
          if (pass == npass - 1) {
            // dQ += dZ_block K_block: the ring region is re-used with the key-major slot geometry now
            // that the Z block's MMAs have drained, and handed back when this block's dQ MMAs have
            const int key0 = kb * 256, keys = min(P, key0 + 256) - key0;
            const int nj = (keys + 31) >> 5;
            const bool lastblk = single && o == nkb - 1;
            for (int k = 0; k < nj && ok; ++k, ++it2) {
              const int j = lastblk ? tc_chunk_last(k, nj, dlo_item) : k;     // the MMA thread's chunk order
              const int slot = it2 % kTcSlots2;
              ok = mbar_wait(&sh->empty2[slot], ((it2 / kTcSlots2) & 1u) ^ 1u, dead);
              if (!ok) break;
              unsigned char* st = stage0 + slot * kTcStage2Bytes;
              mbar_expect_tx(&sh->full2[slot], k2bytes * (x3 ? 2u : 1u));
              bulk_g2s(st, g2_hi + (size_t)(kb * 8 + j) * k2bytes, k2bytes, &sh->full2[slot]);
              if (x3) bulk_g2s(st + 16384, g2_lo + (size_t)(kb * 8 + j) * k2bytes, k2bytes, &sh->full2[slot]);
            }
            if (multi && o + 1 < nkb && ok) ok = mbar_wait(&sh->p2done, (uint32_t)o & 1u, dead);
          }
          ++nz;
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc2 = idesc_bf16(128, Cp, 0, 1);     // dQ: B read MN-major (N = channel)
      const uint32_t dzh = smem_u32(dzhi), dzl = smem_u32(dzlo);
      const uint32_t lbo2 = (uint32_t)Cp8 * 128u;             // 8-key group stride of a key-major chunk
      uint32_t it1 = 0, it2 = 0, nz = 0, dzphase = 0;          // dzphase bit j: parity of the next completion of dzready[j]
      bool ok = true;
      PNCE_TR(8);
      for (int pass = 0; pass < npass && ok; ++pass) {
        for (int o = 0; o < nkb && ok; ++o) {
          const int g = single ? tc_block_at(o, nkb, kbd_item) : o;
          const int kb = MB ? g % nkbi : g;
          const int NB = min(256, Ppad - kb * 256);
          const uint32_t idesc1 = idesc_bf16(128, NB, 0, 0);
          const uint32_t lbo_k = (uint32_t)NB * 16u;          // slab (c/8) stride of a K chunk in smem
          // the previous Z block must have been read out of TMEM.  Pass 1 of two: the epilogue says so (zfree);
          // pass 2 / single pass, block > 0: implied by having consumed every dzready of the previous block.
          if (multi && !single && nz > 0 && (pass == 0 || o == 0)) ok = mbar_wait(&sh->zfree, (nz - 1) & 1u, dead);
          // ---- Z block = Q_half K_block^T ----
          for (int s = 0; s < nstage && ok; ++s, ++it1) {
            const int slot = it1 % nslots1;
            ok = mbar_wait(&sh->full1[slot], (it1 / nslots1) & 1u, dead);
            tc_fence_after();
            const uint32_t st = smem_u32(stage0 + slot * kTcStageBytes);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {                 // 16 channels = 2 slabs per MMA
              const uint64_t a_hi = smem_desc(st + ks * 4096, 2048, 128);
              const uint64_t b_hi = smem_desc(st + kTcOffKhi + ks * 2 * lbo_k, lbo_k, 128);
              mma_bf16(tmem, a_hi, b_hi, idesc1, (s | ks) ? 1u : 0u);
              if (x3) {
                const uint64_t a_lo = smem_desc(st + kTcOffQlo + ks * 4096, 2048, 128);
                const uint64_t b_lo = smem_desc(st + kTcOffKlo + ks * 2 * lbo_k, lbo_k, 128);
                mma_bf16(tmem, a_hi, b_lo, idesc1, 1u);
                mma_bf16(tmem, a_lo, b_hi, idesc1, 1u);
              }
            }
            mma_commit(&sh->empty1[slot]);
          }
          mma_commit(&sh->zfull);
          ++nz;
          if (pass == 0 && kb == 0) PNCE_TR(9);
          if (pass != npass - 1) continue;
          // ---- dQ += dZ_block K_block, one stage per 32 keys, released chunk by chunk by the epilogue ----
          const int key0 = kb * 256, keys = min(P, key0 + 256) - key0;
          const int nj = (keys + 31) >> 5;
          const bool lastblk = single && o == nkb - 1;
          for (int k = 0; k < nj && ok; ++k, ++it2) {
            const int j = lastblk ? tc_chunk_last(k, nj, dlo_item) : k;       // diagonal chunks last (released after the row sums)
            const int slot = it2 % kTcSlots2;
            ok = mbar_wait(&sh->dzready[j], (dzphase >> j) & 1u, dead);   // per-chunk phase: blocks differ in chunk count
            dzphase ^= 1u << j;
            if (ok) ok = mbar_wait(&sh->full2[slot], (it2 / kTcSlots2) & 1u, dead);
            tc_fence_after();
            if (o == 0 && k == 0) PNCE_TR(10);
            const uint32_t st = smem_u32(stage0 + slot * kTcStage2Bytes);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {                 // 16 keys per MMA
              const uint64_t a_hi = smem_desc(dzh + (uint32_t)(j * 2 + ks) * 4096u, 2048, 128);
              const uint64_t b_hi = smem_desc(st + (uint32_t)ks * 2u * lbo2, lbo2, 128);
              mma_bf16(tmem + 256u, a_hi, b_hi, idesc2, (o | k | ks) ? 1u : 0u);
              if (x3) {
                const uint64_t a_lo = smem_desc(dzl + (uint32_t)(j * 2 + ks) * 4096u, 2048, 128);
                const uint64_t b_lo = smem_desc(st + 16384u + (uint32_t)ks * 2u * lbo2, lbo2, 128);
                mma_bf16(tmem + 256u, a_lo, b_hi, idesc2, 1u);
                mma_bf16(tmem + 256u, a_hi, b_lo, idesc2, 1u);
              }
            }
            mma_commit(&sh->empty2[slot]);
          }
          if (multi) mma_commit(&sh->p2done);
        }
      }
      mma_commit(&sh->dqfull);
      PNCE_TR(11);
    }
  } else {
    // ===================== epilogue: thread <-> logits row =====================
    const int q = warp & 3;                                  // TMEM lane quadrant this warp may touch
    const int i = q * 32 + lane;                             // row inside the half
    const int gi = mh * 128 + i;                             // sorted patch slot
    const bool rowok = gi < P;
    const int et = tid - 64;                                 // 0..127
    if (et != 0) tr = nullptr;
    PNCE_TR(0);
    // 1/||k_j|| of every key (kept in global scratch, reloaded per key block) and ||q_i|| of this row;
    // all partial-sum loads are issued up front
    float rownrm;
    {
      float ssq[8];
#pragma unroll
      for (int s = 0; s < 8; ++s)
        ssq[s] = (s < nstage && rowok) ? __ldcg(L.qss + ((size_t)b * nstage + s) * Ppad + gi) : 0.f;
      bool anybad = false;
      for (int j = et; j < (MB ? 0 : Ppad); j += 128) {       // minibatch mode: per key block (tc_mb_key_weights)
        float ssk[8];
#pragma unroll
        for (int s = 0; s < 8; ++s)
          ssk[s] = (s < nstage && j < P) ? __ldcg(L.kss + ((size_t)b * nstage + s) * Ppad + j) : 0.f;
        float ss = 0.f;
#pragma unroll
        for (int s = 0; s < 8; ++s) ss += ssk[s];
        const float nrm = sqrtf(ss);
        const bool bad = !(nrm == nrm);                       // the gather marks non-finite rows with NaN
        anybad |= bad && j < P;
        const float w = (j < P && !bad) ? 1.0f / fmaxf(nrm, kNormEps) : 0.f;
        if (j < 256) invk_s[j] = w;
        if (multi) L.kinv[(size_t)b * Ppad + j] = w;          // both halves' CTAs write identical values
      }
      if (anybad) sh->badk = 1;
      float ss = 0.f;
#pragma unroll
      for (int s = 0; s < 8; ++s) ss += ssq[s];
      rownrm = sqrtf(ss);
      if (rowok && (!MB || L.qinv != nullptr))                 // rows mode carves no qinv
        L.qinv[(size_t)b * P + gi] =
            (rownrm == rownrm) ? (rownrm < kNormEps ? -1.0f / kNormEps : 1.0f / rownrm) : rownrm;
    }
    if (!MB && multi) __threadfence_block();
    asm volatile("bar.sync 1, 128;" ::: "memory");            // publishes invk_s (block 0), kinv and badk
    {
      const bool badq = rowok && !(rownrm == rownrm);
      const float sc = (rowok && !badq) ? 1.0f / fmaxf(rownrm, kNormEps) : 0.f;     // 1 / max(||q_i||, eps)
      const bool noproj = rownrm < kNormEps;
      bool badrow = badq || (sh->badk != 0);                  // minibatch mode: re-read once every key block was seen

      const float inv_tau = 1.0f / p.tau;
      const float a = sc * inv_tau * kLog2e;                  // acc -> logit in log2 units (times 1/||k_j||)
      const float cl = kClamp * kLog2e;
      const bool need_clamp = inv_tau * 1.02f > kClamp;       // |cos| <= 1: the clamp cannot bind otherwise
      const float coef = rowok ? 1.0f / ((float)P * (float)p.B * (float)p.n_layers) : 0.f;
      const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
      const int kbd = gi >> 8;                                // key block holding this row's diagonal
      const int chd = (gi & 255) >> 5;                        // and the chunk inside it (both warp-uniform)
      uint32_t nz = 0;
      PNCE_TR(1);
      float rowloss, s_i, c1;
      const size_t qoff = (((size_t)b * halves + mh) * Cp8 * 16 + (size_t)(i >> 3)) * 64 + (size_t)(i & 7) * 8;
      const __nv_bfloat16* __restrict__ qh = L.qhi + qoff;     // raw q of this row for the dQ epilogue: its slice of the Q blob
      const __nv_bfloat16* __restrict__ ql = (x3 && L.qlo != nullptr) ? L.qlo + qoff : nullptr;
      TcQChunk qa, qb;
      const uint32_t rowoff = (uint32_t)(i >> 3) * 128u + (uint32_t)(i & 7) * 16u;
      TcDiag dg;
      dg.rowok = rowok;
      dg.pass = true;
      dg.d_w = 0.f;
      dg.off = (uint32_t)((gi & 255) >> 3) * 2048u + rowoff + (uint32_t)(gi & 7) * 2u;
      const int kbd_row = (MB ? gb * nkbi : 0) + kbd;         // the same as a global block index
      auto mb_weights = [&](int g) { tc_mb_key_weights<GN>(p, L, g / nkbi, (g % nkbi) * 256, nstage, et, invk_s, &sh->badk); };
      if (single) {
        // ---- ONE pass per key block (P > 256, clamp cannot bind): exp2 once, unnormalised operand, dQ' += E_blk K_blk;
        //      row sums alongside; the block with this item's diagonals last, its diagonal chunks last and released
        //      only once the row sum is complete (the "- I" patch needs it) ----
        float se4[4] = {0.f, 0.f, 0.f, 0.f};
        float s2 = 0.f, ydacc = 0.f;
        bool own_deferred = false;
        for (int o = 0; o < nkb; ++o) {
          const int g = tc_block_at(o, nkb, kbd_item);
          const int kb = MB ? g % nkbi : g;
          const int key0 = kb * 256, keys = min(P, key0 + 256) - key0;
          const int nch = (keys + 31) >> 5;                     // chunks that hold real columns
          const bool lastblk = o == nkb - 1;
          if (MB) {
            mb_weights(g);
          } else if (o > 0 || kb != 0) {                         // swap in this block's 1/||k_j|| (the prologue left block 0's)
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int j = et; j < 256; j += 128) invk_s[j] = (key0 + j < Ppad) ? __ldcg(L.kinv + (size_t)b * Ppad + key0 + j) : 0.f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
          }
          // zfull of this block also means the previous block's dQ MMAs have finished reading the operand region
          mbar_wait(&sh->zfull, nz & 1u, dead);
          ++nz;
          tc_fence_after();
          if (o == 0) PNCE_TR(2);
          if (lastblk) {                                         // the dQ epilogue's first raw-q chunks fly under the last block
            tc_q_load(qa, qh, ql, 0, nstage);
            tc_q_load(qb, qh, ql, 1, nstage);
          }
          const int cd = (g == kbd_row) ? chd : -1;
          uint32_t r0[32], r1[32];
          tmem_ld32(trow + (lastblk ? tc_chunk_last(0, nch, dlo_item) : 0) * 32, r0);
          for (int k = 0; k < nch; k += 2) {
            const int ca = lastblk ? tc_chunk_last(k, nch, dlo_item) : k;
            const int cb = (k + 1 < nch) ? (lastblk ? tc_chunk_last(k + 1, nch, dlo_item) : k + 1) : -2;
            tmem_ld_wait();
            if (cb >= 0) tmem_ld32(trow + cb * 32, r1);
            tc_pass_single(r0, invk_s + ca * 32, a, x3, dzhi, dzlo, (uint32_t)(ca * 4) * 2048u + rowoff, se4, s2);
            if (ca == cd) {
#pragma unroll
              for (int kk = 0; kk < 32; ++kk) ydacc = (kk == lane) ? __uint_as_float(r0[kk]) : ydacc;
            }
            fence_proxy_async_smem();
            if (ca == cd) own_deferred = true;
            else mbar_arrive(&sh->dzready[ca]);                  // 128 arrivals release chunk ca to the MMA thread
            if (cb >= 0) {
              tmem_ld_wait();
              if (k + 2 < nch) tmem_ld32(trow + (lastblk ? tc_chunk_last(k + 2, nch, dlo_item) : k + 2) * 32, r0);
              tc_pass_single(r1, invk_s + cb * 32, a, x3, dzhi, dzlo, (uint32_t)(cb * 4) * 2048u + rowoff, se4, s2);
              if (cb == cd) {
#pragma unroll
                for (int kk = 0; kk < 32; ++kk) ydacc = (kk == lane) ? __uint_as_float(r1[kk]) : ydacc;
              }
              fence_proxy_async_smem();
              if (cb == cd) own_deferred = true;
              else mbar_arrive(&sh->dzready[cb]);
            }
          }
        }
        const float wd = MB ? fmaxf(tc_mb_key_weight<GN>(p, L, gb, rowok ? gi : 0, nstage), 0.f) : __ldcg(L.kinv + (size_t)b * Ppad + (rowok ? gi : 0));
        const float ydr = ydacc * a * wd;                       // diagonal logit (log2 units)
        const float se = (se4[0] + se4[1]) + (se4[2] + se4[3]);
        const float lse2 = lg2f(se);
        if (MB) badrow = badq || (sh->badk != 0);
        rowloss = rowok ? (lse2 - ydr) * kLn2 : 0.f;            // :94, labels = arange
        if (badrow && rowok) rowloss = __int_as_float(0x7fc00000);
        PNCE_TR(3);
        if (own_deferred) {
          // the "- I" term: dQ' = sum_j e_ij k^_j - se_i k^_i, i.e. the operand's diagonal entry becomes
          // (e_ii - se_i) / ||k_i||; this warp's 32 arrivals then release its chunk
          dg.d_w = (ex2f(ydr) - se) * wd;
          tc_fix_diag(dg, x3, dzhi, dzlo);
          fence_proxy_async_smem();
          mbar_arrive(&sh->dzready[chd]);
        }
        s_i = coef * (s2 / se - ydr) * kLn2;                    // sum_j dZ_ij z_ij with dZ = coef (e / se - I)
        c1 = inv_tau * sc * (coef / se);                         // the accumulator holds the unnormalised sum
      } else {
        // ---- pass A: row sum of exp2 over all key blocks, diagonal ----
        float se4[4] = {0.f, 0.f, 0.f, 0.f};
        float ydacc = 0.f;                                      // raw accumulator of the diagonal element
        for (int g = 0; g < nkb; ++g) {
          const int kb = MB ? g % nkbi : g;
          const int key0 = kb * 256, keys = min(P, key0 + 256) - key0;
          const int nch = (keys + 31) >> 5;                     // chunks that hold real columns
          const bool pad = (nch * 32 != keys);                  // the block's last chunk holds padding columns
          if (MB) {
            mb_weights(g);
          } else if (kb > 0) {                                   // swap in this block's 1/||k_j||
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int j = et; j < 256; j += 128) invk_s[j] = (key0 + j < Ppad) ? __ldcg(L.kinv + (size_t)b * Ppad + key0 + j) : 0.f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
          }
          mbar_wait(&sh->zfull, nz & 1u, dead);
          ++nz;
          tc_fence_after();
          if (g == 0) PNCE_TR(2);
          const int cd = (g == kbd_row) ? chd : -1;
          if (need_clamp) tc_row_pass_a<true>(trow, nch, invk_s, a, cl, cd, lane, se4, ydacc, pad);
          else tc_row_pass_a<false>(trow, nch, invk_s, a, cl, cd, lane, se4, ydacc, pad);
          if (multi) {
            tc_fence_before();
            mbar_arrive(&sh->zfree);                             // this Z block may be overwritten
          }
        }
        const float wd = MB ? fmaxf(tc_mb_key_weight<GN>(p, L, gb, rowok ? gi : 0, nstage), 0.f) : multi ? __ldcg(L.kinv + (size_t)b * Ppad + (rowok ? gi : 0)) : invk_s[gi];
        const float ydr = ydacc * a * wd;                       // unclamped diagonal logit (log2 units)
        const float yd = need_clamp ? fminf(fmaxf(ydr, -cl), cl) : ydr;
        const float se = (se4[0] + se4[1]) + (se4[2] + se4[3]);   // padding columns were masked out in pass A
        const float lse2 = lg2f(se);
        if (MB) badrow = badq || (sh->badk != 0);
        rowloss = rowok ? (lse2 - yd) * kLn2 : 0.f;              // :94, labels = arange
        if (badrow && rowok) rowloss = __int_as_float(0x7fc00000);
        PNCE_TR(3);
        // raw q of the first two channel chunks for the dQ epilogue, from this row's slice of the Q operand
        // blob: issued now, so the loads fly under pass B (phase 2 finishes right behind pass B: there is
        // no other slack to hide them in)
        tc_q_load(qa, qh, ql, 0, nstage);
        tc_q_load(qb, qh, ql, 1, nstage);
        // ---- pass B: dZ (pre-divided by ||k_j||) -> smem A operand chunk by chunk, s_i ----
        float s2 = 0.f;
        dg.pass = !need_clamp || fabsf(ydr) <= cl;
        dg.d_w = dg.pass ? (ex2f(yd - lse2) - 1.f) * coef * wd : 0.f;
        for (int g = 0; g < nkb; ++g) {
          const int kb = MB ? g % nkbi : g;
          const int key0 = kb * 256, keys = min(P, key0 + 256) - key0;
          const int nch = (keys + 31) >> 5;
          if (multi) {
            // this block's 1/||k_j||; the Z block is recomputed by the MMA thread (pass 2).  zfull of this
            // block also means the previous block's dQ MMAs have finished reading the dZ operand.
            if (MB) {
              mb_weights(g);
            } else {
              asm volatile("bar.sync 1, 128;" ::: "memory");
              for (int j = et; j < 256; j += 128) invk_s[j] = (key0 + j < Ppad) ? __ldcg(L.kinv + (size_t)b * Ppad + key0 + j) : 0.f;
              asm volatile("bar.sync 1, 128;" ::: "memory");
            }
            mbar_wait(&sh->zfull, nz & 1u, dead);
            ++nz;
            tc_fence_after();
          }
          const int cd = (g == kbd_row) ? chd : -1;
          uint64_t* dzr = sh->dzready;
          if (need_clamp) tc_row_pass_b<true>(trow, nch, invk_s, a, cl, lse2, coef, x3, dzhi, dzlo, rowoff, cd, dg, dzr, s2);
          else tc_row_pass_b<false>(trow, nch, invk_s, a, cl, lse2, coef, x3, dzhi, dzlo, rowoff, cd, dg, dzr, s2);
        }
        if (rowok && dg.pass) s2 = fmaf(-coef, ydr, s2);         // the diagonal's "- I" term of sum_j dZ_ij y_ij
        s_i = s2 * kLn2;                                          // sum_j dZ_ij z_ij
        c1 = inv_tau * sc;
      }
      tc_fence_before();
      PNCE_TR(4);
      // row losses: warp shuffle, then one partial per CTA (deterministic order)
      rowloss = warp_sum(rowloss);
      if (lane == 0) sh->red[q] = rowloss;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (et == 0) L.partial[(size_t)b * L.nparts + mh] = sh->red[0] + sh->red[1] + sh->red[2] + sh->red[3];
      // ---- dQ epilogue: dq/tau -> normalise backward -> dxT (coalesced: lane <-> consecutive slot) ----
      // F.normalize backward: (g - x^(x^.g)) / n when n >= eps, else g / eps
      //   dx = dq*sc - q_raw * (sc^2 s_i)       with dq = acc / tau
      const float c2 = noproj ? 0.f : sc * sc * s_i;
      float* __restrict__ dxrow = L.dxT + (size_t)b * C * Ppad + (rowok ? gi : 0);   // dxpitch == Ppad on this path
      if (p.nhwc) dxrow = L.dxT + ((size_t)b * Ppad + (rowok ? gi : 0)) * C;         // channels-last maps: row-major rows
      PNCE_TR(5);
      // head mode: d loss / d (head output) as a row blob [tile = b*halves+mh][c/8][16][8][8]
      __nv_bfloat16* dyh = L.dyhi ? L.dyhi + qoff : nullptr;
      __nv_bfloat16* dyl = (L.dyhi && L.dylo) ? L.dylo + qoff : nullptr;
      // rows mode (minibatch only): rows used as given -- no normalise backward (c2 = 0), d loss / d q row-major in the
      // caller's row order
      const bool rows = MB && p.rows_mode;
      if (rows) dxrow = L.dq_rows + ((size_t)b * P + (rowok ? gi : 0)) * C;
      if (p.nhwc || rows) tc_dq_epilogue<0>(trow + 256u, nstage, C, qh, ql, dxrow, c1, rows ? 0.f : c2, rowok, dyh, dyl, &sh->dqfull, dead, qa, qb, C, 0u, true);
      else switch (Ppad >> 7) {
        case 1: tc_dq_epilogue<128>(trow + 256u, nstage, C, qh, ql, dxrow, c1, c2, rowok, dyh, dyl, &sh->dqfull, dead, qa, qb); break;
        case 2: tc_dq_epilogue<256>(trow + 256u, nstage, C, qh, ql, dxrow, c1, c2, rowok, dyh, dyl, &sh->dqfull, dead, qa, qb); break;
        default: tc_dq_epilogue<0>(trow + 256u, nstage, C, qh, ql, dxrow, c1, c2, rowok, dyh, dyl, &sh->dqfull, dead, qa, qb, Ppad); break;
      }
      PNCE_TR(6);
      tc_fence_before();
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
  if (tid == 0 && sh->dead) {
    p.counter[1] = 1u;                                        // finalize_losses turns the loss into NaN (in-band)
    if (p.nonfinite != nullptr) *reinterpret_cast<volatile int*>(p.nonfinite + 1) = 1;   // protocol timeout flag (may be mapped host memory)
  }
  if (p.trace != nullptr && tid == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.trace[64 + 3 * (size_t)blockIdx.x + 2] = (long long)t;
  }
  last_cta_finalize<GN>(p, &sh->flag, smem);                   // every CTA-wide phase is over (the __syncthreads above): the ring is free scratch
}

__global__ void __launch_bounds__(kTcThreads, 1) k_loss_tc(const __grid_constant__ Params p,
                                                           const __grid_constant__ BlockMap m) {
  pdl_launch();
  loss_tc_body<false>(p, m);
}

__global__ void __launch_bounds__(kTcThreads, 1) k_loss_tc_mb(const __grid_constant__ Params p,
                                                              const __grid_constant__ BlockMap m) {
  pdl_launch();
  loss_tc_body<true>(p, m);
}

__global__ void __launch_bounds__(kTcThreads, 1) k_loss_tc_mb_gn(const __grid_constant__ Params p,
                                                                 const __grid_constant__ BlockMap m) {
  pdl_launch();
  loss_tc_body<true, true>(p, m);
}

// -------------------------------------------------------------------------------------------------
// Self-test kernel: D(128 x N) = A(128 x K) * B, operands given as pre-tiled blobs with the
// descriptor parameters supplied by the host.  Exercises bulk copy, mbarrier tx, TMEM alloc,
// tcgen05.mma (K-major or MN-major B), commit and tcgen05.ld exactly as k_loss_tc uses them.
// -------------------------------------------------------------------------------------------------
struct ProbeArgs {
  const void* a_blob; const void* b_blob; float* d_out; int* err;
  uint32_t a_bytes, b_bytes;
  uint32_t a_lbo, a_sbo, a_kstep;      // bytes; a_kstep = start-address advance per K=16 step
  uint32_t b_lbo, b_sbo, b_kstep;
  int n, k, b_mn_major;
};

__global__ void __launch_bounds__(128, 1) k_umma_probe(const __grid_constant__ ProbeArgs a) {
  pdl_enter();
  extern __shared__ __align__(1024) unsigned char smem[];
  using namespace umma;
  __shared__ uint64_t full, done;
  __shared__ uint32_t tmem_base;
  __shared__ int dead;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* sa = smem;
  unsigned char* sb = smem + ((a.a_bytes + 1023u) & ~1023u);
  if (tid == 0) {
    mbar_init(&full, 1); mbar_init(&done, 1);
    dead = 0;
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc<256>(&tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base;
  if (tid == 0) {
    mbar_expect_tx(&full, a.a_bytes + a.b_bytes);
    bulk_g2s(sa, a.a_blob, a.a_bytes, &full);
    bulk_g2s(sb, a.b_blob, a.b_bytes, &full);
    if (mbar_wait(&full, 0u, &dead)) {
      tc_fence_after();
      const uint32_t idesc = idesc_bf16(128, a.n, (a.b_mn_major >> 1) & 1, a.b_mn_major & 1);   // bit 0: B, bit 1: A
      for (int ks = 0; ks < a.k / 16; ++ks) {
        const uint64_t da = smem_desc(smem_u32(sa) + ks * a.a_kstep, a.a_lbo, a.a_sbo);
        const uint64_t db = smem_desc(smem_u32(sb) + ks * a.b_kstep, a.b_lbo, a.b_sbo);
        mma_bf16(tmem, da, db, idesc, ks ? 1u : 0u);
      }
    }
    mma_commit(&done);
  }
  __syncwarp();
  const bool ok = mbar_wait(&done, 0u, &dead);
  tc_fence_after();
  for (int ch = 0; ch < a.n / 32; ++ch) {
    uint32_t r[32];
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + ch * 32, r);
    tmem_ld_wait();
#pragma unroll
    for (int k = 0; k < 32; ++k) a.d_out[(size_t)(warp * 32 + lane) * a.n + ch * 32 + k] = __uint_as_float(r[k]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<256>(tmem);
  }
  if (tid == 0 && (!ok || dead)) *a.err = 1;
}

}  // namespace pnce
