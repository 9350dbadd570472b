// Launch 2 of the forward (PNCE_MATH_SIMT_F32): per (layer, image, 32-row tile)
//   Z = Q K^T / tau  ->  clamp  ->  diagonal CE (row reductions by warp shuffle)
//   -> dZ = (softmax - I) * mask / (P B L)  ->  dQ = dZ K / tau  ->  normalise-backward
// and the gradient rows are written as dxT[b][c][rank[p]] (unit upstream gradient).
// The P x P logits live in shared memory only.  Replaces patchnce_cut.py:83-110 and the autograd
// backward of :77-94 (SURVEY.md section 8 rows a8-a11).  The last CTA to finish folds the partial
// row-loss sums into the scalar loss deterministically and applies the non-finite guards.
#pragma once
#include "common.cuh"

namespace pnce {

constexpr int kStageFloats = 288 * 33;   // phase A: K tile 256x33 + Q tile 32x33; C/D reuse it

__host__ __device__ inline size_t loss_simt_smem_bytes(int P) {
  int Pp = (P + 255) & ~255;
  return (size_t)(32 * Pp + kStageFloats + 32 + 8) * sizeof(float);
}

// Deterministic epilogue run by the last CTA of the launch: per-image losses, the reference's
// non-finite guards, batch and layer means.  Parallel over the batch (a block-wide reduction in a
// fixed order per layer) -- a single thread walking L*B values costs one L2 round trip per value,
// ~40 us at B=64, on the critical path of every step.
// GN: global negatives (k_loss_tc_mb_gn) -- the guard of a layer also reads every rank's query flags.
constexpr int kFinalizeScratchBytes = (32 + 32 + PNCE_MAX_LAYERS + 1) * 4;
template <bool GN = false>
__device__ void finalize_losses(const Params& p, void* scratch) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  const int B = p.B, nl = p.n_layers;
  // scratch: kFinalizeScratchBytes of the caller's shared memory (the tcgen05 kernels have no static shared memory to
  // spare: static + dynamic is exactly the 227 KB a CTA may have, and a static array costs a whole 1 KB of alignment)
  float* w_sum = static_cast<float*>(scratch);                  // [32] one slot per warp of ANY launch shape (k_loss_tc_p: 11 warps)
  int* w_bad = reinterpret_cast<int*>(w_sum + 32);              // [32]
  int* layer_bad = w_bad + 32;                                  // [PNCE_MAX_LAYERS]
  int& any_guard = layer_bad[PNCE_MAX_LAYERS];
  float total = 0.f;                                            // thread 0 only
  int bad_total = 0;
  for (int l = 0; l < nl; ++l) {
    const LayerDev& L = p.L[l];
    float acc = 0.f;
    int nbad = 0;
    if (p.mb) {
      // minibatch negatives: the layer is one group of B * P rows -- mean over all of them, and the image guard
      // (:97-99) applied to that single group: a non-finite group contributes 0 and all its rows are guarded
      for (int b = tid; b < B; b += nthr)
        for (int t = 0; t < L.nparts; ++t) acc += __ldcg(L.partial + (size_t)b * L.nparts + t);
      acc = warp_sum(acc);
      if (lane == 0) w_sum[warp] = acc;
      __syncthreads();
      if (tid == 0) {
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w) s += w_sum[w];
        const float sl = s / ((float)L.P * (float)B);
        int bad = isfinite(sl) ? 0 : 1;
        // global negatives: the group is every rank's rows -- a non-finite query row on any rank guards the layer
        for (int w = 0; GN && w < p.kworld; ++w)
          bad |= __ldcg(reinterpret_cast<const int*>(reinterpret_cast<const unsigned char*>(p.qbad) + w * p.kslot) + l) != 0;
        layer_bad[l] = 0;                                       // guarded like an image: NaN rows keep their NaN
        w_bad[0] = bad;
        p.loss_out[1 + l] = bad ? 0.f : sl;
        total += bad ? 0.f : sl;
        bad_total += bad;                                       // nonfinite[0] counts guarded layers in this mode
      }
      __syncthreads();
      const int bad = w_bad[0];
      for (int b = tid; b < B; b += nthr) {
        p.lossimg[l * B + b] = 0.f;
        p.valid[l * B + b] = bad ? 0 : 1;
      }
      __syncthreads();
      continue;
    }
    for (int b = tid; b < B; b += nthr) {
      float s = 0.f;
      for (int t = 0; t < L.nparts; ++t) s += __ldcg(L.partial + (size_t)b * L.nparts + t);
      const float lb = s / (float)L.P;                          // CE reduction='mean' over rows  :94
      const int ok = isfinite(lb) ? 1 : 0;                      // :97
      p.lossimg[l * B + b] = ok ? lb : 0.f;                     // :99
      p.valid[l * B + b] = ok;
      acc += ok ? lb : 0.f;                                     // :101
      nbad += ok ? 0 : 1;
    }
    acc = warp_sum(acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nbad += __shfl_xor_sync(0xffffffffu, nbad, o);
    if (lane == 0) { w_sum[warp] = acc; w_bad[warp] = nbad; }
    __syncthreads();
    if (tid == 0) {
      float sl = 0.f;
      int nb = 0;
      for (int w = 0; w < nwarp; ++w) { sl += w_sum[w]; nb += w_bad[w]; }
      sl = sl / (float)B;                                       // :103
      layer_bad[l] = isfinite(sl) ? 0 : 1;                      // :106-108
      if (layer_bad[l]) sl = 0.f;
      p.loss_out[1 + l] = sl;
      total += sl;                                              // :38
      bad_total += nb + layer_bad[l];
    }
    __syncthreads();
  }
  if (tid == 0) {
    p.loss_out[0] = total / (float)nl;                          // :40
    // a tcgen05 pipeline that timed out (umma::mbar_wait) left garbage behind: say so in the value itself
    if (__ldcg(p.counter + 1) != 0u) p.loss_out[0] = __int_as_float(0x7fc00000);
    int nb = 0;
    for (int l = 0; l < nl; ++l) nb += layer_bad[l];
    if (p.nonfinite) *p.nonfinite = bad_total - nb;             // images guarded (layer guards are not counted)
    any_guard = bad_total > 0;
  }
  __syncthreads();
  if (!any_guard) return;                                       // the common case: nothing to overwrite
  // Guarded images receive an exactly-zero upstream gradient; autograd still pushes it through the
  // normalise backward, so rows holding NaN/Inf come out NaN and everything else 0 (see oracle).
  for (int l = 0; l < nl; ++l) {
    const LayerDev& L = p.L[l];
    for (int b = 0; b < B; ++b) {
      if (p.valid[l * B + b] && !layer_bad[l]) continue;
      const size_t n = (size_t)L.C * L.P;
      if (L.dq_rows != nullptr) {
        for (size_t i = tid; i < n; i += nthr) L.dq_rows[(size_t)b * n + i] = 0.f;
      } else if (L.dyhi != nullptr) {
        // head mode: the image's rows of the d loss / d Y blob (zero upstream gradient)
        const size_t per = (size_t)L.Ppad * L.Cp;
        for (size_t i = tid; i < per; i += nthr) {
          L.dyhi[(size_t)b * per + i] = __float2bfloat16_rn(0.f);
          if (L.dylo != nullptr) L.dylo[(size_t)b * per + i] = __float2bfloat16_rn(0.f);
        }
      } else {
        for (size_t i = tid; i < n; i += nthr) {
          int c = (int)(i / L.P), pp = (int)(i % L.P);
          float inv = L.qinv[(size_t)b * L.P + pp];
          float v = (!layer_bad[l] && !(inv == inv)) ? __int_as_float(0x7fc00000) : 0.f;
          const int slot = L.sorted ? pp : L.rank[pp];
          if (p.nhwc) L.dxT[((size_t)b * L.dxpitch + slot) * L.C + c] = v;        // row-major rows (channels-last maps)
          else L.dxT[((size_t)b * L.C + c) * L.dxpitch + slot] = v;
        }
      }
    }
  }
}

template <bool GN = false>
__device__ __forceinline__ void last_cta_finalize(const Params& p, int* flag_s, void* scratch) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = atomicAdd(p.counter, 1u);
    *flag_s = (t == p.total_ctas - 1) ? 1 : 0;
  }
  __syncthreads();
  if (*flag_s) {
    __threadfence();
    finalize_losses<GN>(p, scratch);
    if (threadIdx.x == 0) { p.counter[0] = 0u; p.counter[1] = 0u; }
  }
}

__global__ void __launch_bounds__(kThreads) k_loss_simt(const __grid_constant__ Params p,
                                                        const __grid_constant__ BlockMap m) {
  pdl_enter();
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  const int l = find_layer(m, blockIdx.x, p.n_layers);
  const LayerDev& L = p.L[l];
  const int local = (int)(blockIdx.x - m.start[l]);
  const int tile = local % L.ntiles, b = local / L.ntiles;
  const int P = L.P, C = L.C;
  const int Pp = (P + 255) & ~255;
  float* zs = sm;                      // [32][Pp] raw logits, then dZ
  float* stage = sm + 32 * Pp;         // kStageFloats
  float* rl = stage + kStageFloats;    // [32] row losses
  int* flag_s = reinterpret_cast<int*>(rl + 32);
  const int row0 = tile * kRowTile;
  const float* qn = L.qn + (size_t)b * P * C;
  const float* kn = L.kn + (size_t)b * P * C;
  const float tau = p.tau;

  // ---- phase A: raw logits tile (32 x P) = Q_tile K^T / tau ---------------------------------
  {
    float* Ks = stage;                 // [256][33]
    float* Qs = stage + 256 * 33;      // [32][33]
    for (int ct = 0; ct < Pp; ct += 256) {
      float acc[4][8];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int n = 0; n < 8; ++n) acc[r][n] = 0.f;
      for (int c0 = 0; c0 < C; c0 += 32) {
        for (int e = tid; e < 32 * 32; e += kThreads) {
          int r = e >> 5, kk = e & 31, i = row0 + r, c = c0 + kk;
          Qs[r * 33 + kk] = (i < P && c < C) ? qn[(size_t)i * C + c] : 0.f;
        }
        for (int e = tid; e < 256 * 32; e += kThreads) {
          int j = e >> 5, kk = e & 31, jj = ct + j, c = c0 + kk;
          Ks[j * 33 + kk] = (jj < P && c < C) ? kn[(size_t)jj * C + c] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 32; ++kk) {
          float q[4], k[8];
#pragma unroll
          for (int r = 0; r < 4; ++r) q[r] = Qs[(ty * 4 + r) * 33 + kk];
#pragma unroll
          for (int n = 0; n < 8; ++n) k[n] = Ks[(tx + 32 * n) * 33 + kk];
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int n = 0; n < 8; ++n) acc[r][n] = fmaf(q[r], k[n], acc[r][n]);
        }
        __syncthreads();
      }
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int n = 0; n < 8; ++n) zs[(ty * 4 + r) * Pp + ct + tx + 32 * n] = acc[r][n] / tau;   // :85
    }
  }
  __syncthreads();

  // ---- phase B: diagonal CE per row (warp = 4 rows, lanes = columns) -------------------------
  const float coef = 1.0f / ((float)P * (float)p.B * (float)p.n_layers);
  float si[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int row = ty * 4 + r, i = row0 + row;
    float* zr = zs + row * Pp;
    float rowloss = 0.f, s_i = 0.f;
    if (i < P) {
      float mx = -INFINITY;
      for (int j = tx; j < P; j += 32) mx = fmaxf(mx, clamp_nan(zr[j], kClamp));      // :88
      mx = warp_max(mx);
      float se = 0.f;
      for (int j = tx; j < P; j += 32) se += expf(clamp_nan(zr[j], kClamp) - mx);
      se = warp_sum(se);
      const float lse = mx + logf(se);
      rowloss = lse - clamp_nan(zr[i], kClamp);                                        // :94, labels = arange
      for (int j = tx; j < Pp; j += 32) {
        float d = 0.f;
        if (j < P) {
          const float zraw = zr[j];
          const float pj = expf(clamp_nan(zraw, kClamp) - lse);
          const bool pass = (zraw >= -kClamp) && (zraw <= kClamp);                     // clamp backward
          d = pass ? (pj - (j == i ? 1.f : 0.f)) * coef : 0.f;
          s_i = fmaf(d, zraw, s_i);            // q_hat . dq  ==  sum_j dZ_ij * zraw_ij
        }
        zr[j] = d;
      }
      s_i = warp_sum(s_i);
    } else {
      for (int j = tx; j < Pp; j += 32) zr[j] = 0.f;
    }
    si[r] = s_i;
    if (tx == 0) rl[row] = rowloss;
  }
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
    for (int r = 0; r < 32; ++r) s += rl[r];
    L.partial[(size_t)b * L.nparts + tile] = s;
  }

  // ---- phase C/D: dQ tile = dZ K / tau, normalise backward, transposed store -----------------
  for (int cb = 0; cb < C; cb += 256) {
    float acc[4][8];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int n = 0; n < 8; ++n) acc[r][n] = 0.f;
    float* Kc = stage;                 // [32][256]
    for (int j0 = 0; j0 < P; j0 += 32) {
      for (int e = tid; e < 32 * 256; e += kThreads) {
        int jj = e >> 8, cc = e & 255, j = j0 + jj, c = cb + cc;
        Kc[jj * 256 + cc] = (j < P && c < C) ? kn[(size_t)j * C + c] : 0.f;
      }
      __syncthreads();
#pragma unroll 8
      for (int jj = 0; jj < 32; ++jj) {
        float d[4], k[8];
#pragma unroll
        for (int r = 0; r < 4; ++r) d[r] = zs[(ty * 4 + r) * Pp + j0 + jj];
#pragma unroll
        for (int n = 0; n < 8; ++n) k[n] = Kc[jj * 256 + tx + 32 * n];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int n = 0; n < 8; ++n) acc[r][n] = fmaf(d[r], k[n], acc[r][n]);
      }
      __syncthreads();
    }
    if (L.dq_rows != nullptr) {
      // rows API: d loss / d q_hat in (B*P, D) layout, coalesced along c
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int i = row0 + ty * 4 + r;
        if (i < P) {
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            const int c = cb + tx + 32 * n;
            if (c < C) L.dq_rows[((size_t)b * P + i) * C + c] = acc[r][n] / tau;
          }
        }
      }
    } else {
      float* St = stage;               // [256][33] : dx tile transposed
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int i = row0 + ty * 4 + r;
        const float inv = (i < P) ? L.qinv[(size_t)b * P + i] : 0.f;
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          const int c = cb + tx + 32 * n;
          float dx = 0.f;
          if (i < P && c < C) {
            const float dq = acc[r][n] / tau;
            const float qh = qn[(size_t)i * C + c];
            // F.normalize backward: (g - x^(x^.g)) / n  when n >= eps, else g / eps
            dx = (inv < 0.f) ? dq * (-inv) : (dq - qh * si[r]) * inv;
          }
          St[(tx + 32 * n) * 33 + ty * 4 + r] = dx;
        }
      }
      __syncthreads();
      {
        const int i = row0 + tx;
        const int slot = (i < P) ? L.rank[i] : 0;
        for (int cc = ty; cc < 256; cc += 8) {
          const int c = cb + cc;
          if (c < C && i < P) L.dxT[((size_t)b * C + c) * L.dxpitch + slot] = St[cc * 33 + tx];
        }
      }
      __syncthreads();
    }
  }

  last_cta_finalize(p, flag_s, sm);                            // every phase is over: the logits tile is free scratch
}

}  // namespace pnce
