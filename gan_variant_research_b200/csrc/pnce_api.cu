// libpnce.so -- C ABI (include/pnce.h) over the sm_100a kernels.  Host side only: argument checks,
// workspace carving, launch geometry.  No device allocation, no host sync, graph-capturable.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "dense.cuh"
#include "gather.cuh"
#include "gather_tc.cuh"
#include "gemm_tc.cuh"
#include "gemm_tc_persist.cuh"
#include "loss_simt.cuh"
#include "loss_tc.cuh"
#include "loss_tc_persist.cuh"
#include "nhwc.cuh"
#include "netf.cuh"
#include "rows_pack.cuh"
#include "multi_tensor.cuh"
#include "sample_bwd.cuh"
#include "dside.cuh"
#include "comp_alloc.cuh"

namespace pnce {

static thread_local char g_cuda_err[256] = "";

static int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
  return PNCE_ERR_CUDA;
}
#define PNCE_CUDA(call)                                  \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static size_t dtype_size(int dtype) { return dtype == PNCE_F32 ? 4 : 2; }

// Carves the workspace.  With base == nullptr only the size is computed.
struct Carver {
  unsigned char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<unsigned char*>(b)) {}
  template <typename T> T* take(size_t n) {
    off = align_up(off, 256);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

static int check_layers(const pnce_layer_t* layers, int n_layers, int B) {
  if (layers == nullptr || n_layers < 1 || B < 1) return PNCE_ERR_ARG;
  if (n_layers > PNCE_MAX_LAYERS) return PNCE_ERR_UNSUPPORTED;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    if (a.C < 1 || a.H < 1 || a.W < 1 || a.P < 1) return PNCE_ERR_ARG;
    if ((long long)a.H * a.W > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
    if (a.P > PNCE_MAX_PATCHES || a.C > PNCE_MAX_CHANNELS) return PNCE_ERR_UNSUPPORTED;
  }
  return PNCE_OK;
}

static bool tc_shapes_ok(const pnce_layer_t* layers, int n_layers) {
  for (int l = 0; l < n_layers; ++l)
    if (layers[l].P > 1024 || layers[l].C > 256) return false;
  return true;
}

// minibatch negatives: the tensor-core envelope, and at most 65536 keys (B * Ppad) per layer -- the bound under which the
// single-pass row sum (no running maximum) stays finite in fp32
static constexpr long long kMbMaxKeys = 65536;
static bool mb_keys_ok(int B, int P) { return (long long)B * ((P + 127) / 128 * 128) <= kMbMaxKeys; }
static bool mb_shapes_ok(const pnce_layer_t* layers, int n_layers, int B) {
  if (!tc_shapes_ok(layers, n_layers)) return false;
  for (int l = 0; l < n_layers; ++l)
    if (!mb_keys_ok(B, layers[l].P)) return false;
  return true;
}

// global negatives: the envelope of the GLOBAL batch of world * batch_local images -- the product must fit an int, then
// pass the route's shape test (a status: PNCE_OK, or the code to return)
template <typename ShapeTest>
static int global_batch_check(int world, int batch_local, ShapeTest shapes) {
  if ((long long)world * batch_local > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  return shapes(world * batch_local);
}

// Fills Params (pointers into the workspace) for the fused path; returns bytes used.
// tc = carve the tensor-core operand blobs instead of the fp32 normalised rows.
// The id bookkeeping of every layer (k_prep's outputs): sid, perm, rank, cslot.  It lives at the head of the
// workspace, or -- pnce_plan_ids / pnce_fwd_planned -- in a buffer of its own, so that the id sort can run on
// another stream before the workspace of the step even exists.  With base == nullptr only the size is computed.
static size_t carve_plan(const pnce_layer_t* layers, int n_layers, void* base, Params* p) {
  Carver cv(base);
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    const int HW = a.H * a.W;
    int* sid = cv.take<int>(a.P);
    int* perm = cv.take<int>(a.P);
    int* rank = cv.take<int>(a.P);
    int* cslot = cv.take<int>((size_t)(HW + kTilePos - 1) / kTilePos + 1);
    if (p != nullptr) {
      LayerDev& L = p->L[l];
      L.sid = sid; L.perm = perm; L.rank = rank; L.cslot = cslot;
    }
  }
  return align_up(cv.off, 256);
}

static size_t carve_fused(const pnce_layer_t* layers, int n_layers, int B, bool tc, bool x3, void* ws,
                          Params* out, void* plan = nullptr) {
  Carver cv(ws);
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n_layers;
  p.B = B;
  p.counter = cv.take<unsigned>(64);
  p.lossimg = cv.take<float>((size_t)n_layers * B);
  p.valid = cv.take<int>((size_t)n_layers * B);
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    LayerDev& L = p.L[l];
    L.src = a.src; L.tgt = a.tgt; L.dtgt = a.dtgt;
    L.ids = reinterpret_cast<const long long*>(a.ids);
    L.C = a.C; L.HW = a.H * a.W; L.P = a.P;
    L.nwords = (L.HW + 31) / 32;
    L.ntiles = (L.P + kRowTile - 1) / kRowTile;
    const size_t rows = (size_t)B * a.P * a.C;
    if (plan == nullptr) {
      L.sid = cv.take<int>(a.P);
      L.perm = cv.take<int>(a.P);
      L.rank = cv.take<int>(a.P);
      L.cslot = cv.take<int>((size_t)(L.HW + kTilePos - 1) / kTilePos + 1);
    }
    L.qinv = cv.take<float>((size_t)B * a.P);
    L.dxpitch = tc ? (a.P + 127) / 128 * 128 : a.P;
    L.dxT = cv.take<float>((size_t)B * a.C * L.dxpitch);
    L.dq_rows = nullptr;
    if (!tc) {
      L.nparts = L.ntiles;
      L.qn = cv.take<float>(rows);
      L.kn = cv.take<float>(rows);
    } else {
      L.sorted = 1;
      L.Cp = (a.C + 31) / 32 * 32;
      L.Ppad = (a.P + 127) / 128 * 128;
      L.nchunk = L.Cp / 32;
      L.nparts = L.Ppad / 128;
      const size_t blob = (size_t)B * L.Ppad * L.Cp;
      L.qhi = cv.take<__nv_bfloat16>(blob);
      L.khi = cv.take<__nv_bfloat16>(blob);
      if (x3) {
        L.qlo = cv.take<__nv_bfloat16>(blob);
        L.klo = cv.take<__nv_bfloat16>(blob);
      }
      L.k2hi = cv.take<__nv_bfloat16>(blob);
      if (x3) L.k2lo = cv.take<__nv_bfloat16>(blob);
      L.qss = cv.take<float>((size_t)B * L.nchunk * L.Ppad);
      L.kss = cv.take<float>((size_t)B * L.nchunk * L.Ppad);
      L.kinv = cv.take<float>((size_t)B * L.Ppad);
    }
    L.partial = cv.take<float>((size_t)B * (L.ntiles > 2 ? L.ntiles : 2));
  }
  if (plan != nullptr) carve_plan(layers, n_layers, plan, &p);
  if (out) *out = p;
  return align_up(cv.off, 256);
}

static size_t gather_smem_bytes(const Params& p, bool with_prep) {
  size_t need = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    size_t g = ((size_t)kRowTile * (p.L[l].C + 1) + 544) * sizeof(float);
    if (g > need) need = g;
    if (with_prep) {
      int n2 = 1;
      while (n2 < p.L[l].P) n2 <<= 1;
      size_t s = (size_t)n2 * 8 + 64;
      if (s > need) need = s;
    }
  }
  return need;
}

// Every kernel of the library is launched through launch_k: with programmatic dependent launch allowed (the default;
// PNCE_PDL=0 in the environment turns it off, read once per process) the launch carries
// cudaLaunchAttributeProgrammaticStreamSerialization, every kernel starts with pdl_enter() (common.cuh: signal the
// dependents, then wait for the prerequisite grids before the first global access), so along one stream the next
// kernel's CTAs are dispatched while the previous grid drains instead of after it has retired -- the launch and
// scheduling latency between the kernels of a step (2-4 us per boundary; a B = 8 step has four kernels of 7-60 us)
// disappears, and results cannot change: no kernel touches memory before its predecessors have completed.
static int pdl_allowed() {
  static const int v = [] {
    const char* e = getenv("PNCE_PDL");
    return e != nullptr ? atoi(e) : 23;   // bit 8 is unused: see SITE 0 below
  }();
  return v;
}

// PNCE_FOLD_PREP=0: always launch k_prep (A/B of the folded id prep, gather_tc.cuh)
static bool pnce_fold_allowed() {
  static const bool v = [] {
    const char* e = getenv("PNCE_FOLD_PREP");
    return !(e != nullptr && e[0] == '0');
  }();
  return v;
}

// SITE: 1 id prep, 2 gather, 4 loss, 16 everything else; PNCE_PDL is a mask over the sites (default: all of them).  SITE 0 =
// the dense-backward kernels (k_dense_*, k_fill_zero, k_scatter_nhwc): ALWAYS launched the ordinary way, and they are the
// only kernels without pdl_enter().  With the attribute on them the NEXT step's gather ran 30 % slower from B = 8 on
// (DESIGN.md 4.9: measured, mechanism not identified), they have nothing to gain -- their predecessor is the persistent
// loss kernel, whose CTAs hold every SM until they exit -- and the two instructions themselves cost k_fill_zero 8 % (393 216
// CTAs of a few dozen instructions each: 378 -> 407 us at B = 64).
template <int SITE = 16, typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = (pdl_allowed() & SITE) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Opt a kernel in to more than 48 KB of dynamic shared memory.  The attribute is sticky per kernel and
// device: what has been set is remembered so the driver call is made once, not per launch.
struct SmemOptIn { const void* fn; int dev; size_t bytes; };
static thread_local SmemOptIn g_optin[64];
static thread_local int g_noptin = 0;

template <typename K> static int set_smem(K kernel, size_t bytes) {
  if (bytes <= 48 * 1024) return PNCE_OK;
  if (bytes > 227 * 1024) return PNCE_ERR_UNSUPPORTED;
  int dev = 0;
  PNCE_CUDA(cudaGetDevice(&dev));
  const void* fn = reinterpret_cast<const void*>(kernel);
  SmemOptIn* e = nullptr;
  for (int i = 0; i < g_noptin; ++i)
    if (g_optin[i].fn == fn && g_optin[i].dev == dev) e = &g_optin[i];
  if (e != nullptr && e->bytes >= bytes) return PNCE_OK;
  PNCE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  if (e == nullptr && g_noptin < 64) e = &g_optin[g_noptin++];
  if (e != nullptr) { e->fn = fn; e->dev = dev; e->bytes = bytes; }
  return PNCE_OK;
}

static int launch_gather(const Params& p, int n_prep, cudaStream_t st) {
  BlockMap m;
  memset(&m, 0, sizeof(m));
  long long acc = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    m.start[l] = acc;
    const long long sides = 2 - p.side0;
    acc += sides * p.B * p.L[l].ntiles;
  }
  m.start[p.n_layers] = acc;
  const size_t smem = gather_smem_bytes(p, n_prep > 0);
  int rc = set_smem(k_gather_prep, smem);
  if (rc != PNCE_OK) return rc;
  if (acc + n_prep > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  launch_k<2>(k_gather_prep, (unsigned)(acc + n_prep), kThreads, smem, st, p, m);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int launch_loss_simt(const Params& p, cudaStream_t st) {
  BlockMap m;
  memset(&m, 0, sizeof(m));
  long long acc = 0;
  size_t smem = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    m.start[l] = acc;
    acc += (long long)p.B * p.L[l].ntiles;
    size_t s = loss_simt_smem_bytes(p.L[l].P);
    if (s > smem) smem = s;
  }
  m.start[p.n_layers] = acc;
  int rc = set_smem(k_loss_simt, smem);
  if (rc != PNCE_OK) return rc;
  if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  Params q = p;
  q.total_ctas = (unsigned)acc;
  launch_k<4>(k_loss_simt, (unsigned)acc, kThreads, smem, st, q, m);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int launch_prep(const Params& p, cudaStream_t st) {
  size_t smem = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    int n2 = 1;
    while (n2 < p.L[l].P) n2 <<= 1;
    const size_t s = (size_t)n2 * 8 + 64;
    if (s > smem) smem = s;
  }
  launch_k<1>(k_prep, (unsigned)p.n_layers, kThreads, smem, st, p);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

#ifdef PNCE_EXPERIMENTS
static int g_gather_in_layer_order = 0;   // experiment knob 8
#else
static constexpr int g_gather_in_layer_order = 0;
#endif

// NCHW gather CTAs of the whole batch, and whether the id prep is folded into them (gather_tc.cuh: k_gather_tc_fold)
static long long gather_tc_ctas(const Params& p, int images) {
  long long acc = 0;
  for (int l = 0; l < p.n_layers; ++l)
    acc += (long long)(2 - p.side0) * images * ((p.L[l].Ppad + 255) / 256) * p.L[l].nchunk;
  return acc;
}
static long long gather_nhwc_ctas(const Params& p, int images) {
  long long acc = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    const long long items = (long long)(2 - p.side0) * images * (p.L[l].Ppad >> 3) * p.L[l].nchunk;
    acc += (items + 8 * kNhwcItemsPerWarp - 1) / (8 * kNhwcItemsPerWarp);
  }
  return acc;
}
static bool gather_tc_folds(const Params& p) {
  return pnce_fold_allowed() && (p.nhwc ? gather_nhwc_ctas(p, p.B) : gather_tc_ctas(p, p.B)) <= kFoldMaxCtas;
}
static size_t fold_smem_bytes(const Params& p) {
  size_t smem = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    int n2 = 1;
    while (n2 < p.L[l].P) n2 <<= 1;
    const size_t b = (size_t)n2 * 8 + 64;
    if (b > smem) smem = b;
  }
  return smem;
}

static int launch_gather_tc(const Params& p, cudaStream_t st, bool fold = false) {
  BlockMap m;
  memset(&m, 0, sizeof(m));
  // light layers (small C) first, heavy layers last: the loss kernel starts with the heavy layers, whose
  // operand blobs are then the most recently written lines in L2 (its first items otherwise start on cold DRAM)
  int order[PNCE_MAX_LAYERS];
  for (int l = 0; l < p.n_layers; ++l) order[l] = l;
  if (!g_gather_in_layer_order)
    for (int i = 1; i < p.n_layers; ++i)
      for (int j = i; j > 0 && p.L[order[j]].C <= p.L[order[j - 1]].C; --j) { int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
  long long acc = 0;
  if (p.nhwc) {
    // channels-last maps: warp items (side, image, 8 slots, 32-channel chunk), 8 warps per CTA, kNhwcItemsPerWarp each
    for (int s = 0; s < p.n_layers; ++s) {
      m.start[s] = acc;
      m.layer[s] = order[s];
      const long long items = (long long)(2 - p.side0) * p.bn * (p.L[order[s]].Ppad >> 3) * p.L[order[s]].nchunk;
      if (items > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;   // the kernel's item arithmetic is 32-bit
      acc += (items + 8 * kNhwcItemsPerWarp - 1) / (8 * kNhwcItemsPerWarp);
    }
    m.start[p.n_layers] = acc;
    if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
    if (fold) launch_k<2>(k_gather_tc_nhwc_fold, (unsigned)acc, kThreads, fold_smem_bytes(p), st, p, m);
    else launch_k<2>(k_gather_tc_nhwc, (unsigned)acc, kThreads, 0, st, p, m);
    PNCE_CUDA(cudaGetLastError());
    return PNCE_OK;
  }
  for (int s = 0; s < p.n_layers; ++s) {
    m.start[s] = acc;
    m.layer[s] = order[s];
    acc += (long long)(2 - p.side0) * p.bn * ((p.L[order[s]].Ppad + 255) / 256) * p.L[order[s]].nchunk;
  }
  m.start[p.n_layers] = acc;
  if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  if (fold) {
    launch_k<2>(k_gather_tc_fold, (unsigned)acc, kThreads, fold_smem_bytes(p), st, p, m);
  } else {
    launch_k<2>(k_gather_tc, (unsigned)acc, kThreads, 0, st, p, m);
  }
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

// Experiment knobs.  The shipped library is built WITHOUT -DPNCE_EXPERIMENTS: the knobs are then compile-time
// constants at their defaults and neither pnce_debug_* nor the experiment kernels exist in libpnce.so (every
// exported symbol is declared in include/pnce.h).  `PNCE_EXPERIMENTS=1 python -m gan_variant_research_b200.build`
// builds libpnce_exp.so with the hooks for the scripts under scratch/.  0 = library default.
struct DebugKnobs {
  int dense_flags = 0;       // bit 0: skip the patch phase (fill ceiling)
  int fwd_chunks = 0;        // n > 1: cut the tensor-core forward into n chunks, loss(c) on an aux stream || gather(c+1)
  int no_persist = 0;        // 1: one CTA per item (k_loss_tc) even where the persistent kernel applies
  int persist_ctas = 0;      // > 0: grid of the persistent loss kernel (default: one CTA per SM)
  long long* trace = nullptr;
  cudaEvent_t post_gather_event = nullptr;   // recorded on the caller's stream between the gather and the loss kernel
  int loss_repeat = 0;       // n > 0: launch the loss kernel n extra times first (is its start-up cost cache coldness?)
  int gemm_dbg = 0;          // head GEMM epilogue: 1 = no global stores, 2 = empty (where does a launch's time go?)
  long long loss_rot = 0;    // persistent loss kernel: 0 = a third of the CTAs start on light items (auto), -1 = plain heavy-first order, n > 0 = rotate by n
};
#ifdef PNCE_EXPERIMENTS
static DebugKnobs g_dbg;
#else
static constexpr DebugKnobs g_dbg{};
#endif

static int sm_count(int* out) {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  PNCE_CUDA(cudaGetDevice(&dev));
  if (dev != cached_dev) {
    PNCE_CUDA(cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev));
    cached_dev = dev;
  }
  *out = cached;
  return PNCE_OK;
}

static int launch_loss_tc(const Params& p, cudaStream_t st, bool single_launch = true) {
  BlockMap m;
  memset(&m, 0, sizeof(m));
  // heavy layers (large C) first: the last, partially filled wave of CTAs is then made of the cheap ones
  int order[PNCE_MAX_LAYERS];
  for (int l = 0; l < p.n_layers; ++l) order[l] = l;
  for (int i = 1; i < p.n_layers; ++i)
    for (int j = i; j > 0 && p.L[order[j]].C > p.L[order[j - 1]].C; --j) { int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
  long long acc = 0;
  for (int s = 0; s < p.n_layers; ++s) {
    m.start[s] = acc;
    m.layer[s] = order[s];
    acc += (long long)p.bn * (p.L[order[s]].Ppad / 128);
  }
  m.start[p.n_layers] = acc;
  if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  if (p.mb) {                                                  // minibatch negatives: one CTA per item, every key block
    auto kernel = p.kworld > 0 ? k_loss_tc_mb_gn : k_loss_tc_mb;   // global negatives: keys from every rank's slot
    int rc = set_smem(kernel, kTcSmemBytes);
    if (rc != PNCE_OK) return rc;
    launch_k<4>(kernel, (unsigned)acc, kTcThreads, kTcSmemBytes, st, p, m);
    PNCE_CUDA(cudaGetLastError());
    return PNCE_OK;
  }
  // P <= 256 everywhere (one key block per item): persistent kernel, one CTA per SM walking the item list
  bool persist = single_launch && !g_dbg.no_persist;
  for (int l = 0; l < p.n_layers; ++l)
    if (p.L[l].Ppad > 256) persist = false;
  if (persist) {
    int nsm = 0;
    int rc = sm_count(&nsm);
    if (rc != PNCE_OK) return rc;
    long long grid = g_dbg.persist_ctas > 0 ? g_dbg.persist_ctas : nsm;
    if (grid > acc) grid = acc;
    rc = set_smem(k_loss_tc_p, kTpSmemBytes);
    if (rc != PNCE_OK) return rc;
    Params q = p;
    q.total_ctas = (unsigned)grid;
    // rotate the item list so that a third of the CTAs starts on an item of the lightest layers (tp_decode), taken
    // from the END of the heavy-first order; an even count keeps the two halves of an image together
    long long rot = 0;
    if (g_dbg.loss_rot == 0) {
      int cmin = p.L[order[p.n_layers - 1]].C;
      long long light = 0;
      for (int sl = p.n_layers - 1; sl >= 0 && p.L[order[sl]].C == cmin; --sl) light += m.start[sl + 1] - m.start[sl];
      rot = light < grid / 3 ? light : grid / 3;
      rot &= ~1LL;
      if (light == acc) rot = 0;                                // one kind of item only: nothing to reorder
    } else if (g_dbg.loss_rot > 0) {
      rot = g_dbg.loss_rot < acc ? g_dbg.loss_rot : 0;
    }
    m.start[PNCE_MAX_LAYERS + 1] = rot > 0 ? acc - rot : 0;
    launch_k<4>(k_loss_tc_p, (unsigned)grid, kTpThreads, kTpSmemBytes, st, q, m);
    PNCE_CUDA(cudaGetLastError());
    return PNCE_OK;
  }
  int rc = set_smem(k_loss_tc, kTcSmemBytes);
  if (rc != PNCE_OK) return rc;
  launch_k<4>(k_loss_tc, (unsigned)acc, kTcThreads, kTcSmemBytes, st, p, m);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}


// ---- chunked tensor-core forward ---------------------------------------------------------------
// The gather is HBM-bound and the tcgen05 loss kernel is not, so the batch is cut into chunks and
// loss(chunk c) runs on an auxiliary stream while gather(chunk c+1) runs on the caller's stream:
//   st : prep, gather(0), gather(1), ...            aux: loss(0), loss(1), ...   (loss(c) after gather(c))
// Fork/join with events only -- no host sync, and the pattern is CUDA-graph capturable.
struct AuxStreams {
  cudaStream_t aux = nullptr;
  cudaEvent_t ev[16] = {};
  cudaEvent_t join = nullptr;
  int device = -1;
};
static thread_local AuxStreams g_aux;

static int aux_streams(AuxStreams** out) {
  int dev = 0;
  PNCE_CUDA(cudaGetDevice(&dev));
  if (g_aux.aux == nullptr || g_aux.device != dev) {
    int lo = 0, hi = 0;
    PNCE_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    PNCE_CUDA(cudaStreamCreateWithPriority(&g_aux.aux, cudaStreamNonBlocking, hi));
    for (auto& e : g_aux.ev) PNCE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    PNCE_CUDA(cudaEventCreateWithFlags(&g_aux.join, cudaEventDisableTiming));
    g_aux.device = dev;
  }
  *out = &g_aux;
  return PNCE_OK;
}

static int forward_tc(Params& p, cudaStream_t st, bool planned = false) {
  int rc = PNCE_OK;
  // planned: pnce_plan_ids has run k_prep already (gather CTA 0 resets the counter); small problems: the gather CTAs
  // sort the ids themselves (k_gather_tc_fold), no k_prep launch
  const bool fold = !planned && (g_dbg.fwd_chunks <= 1 || p.mb) && gather_tc_folds(p);
  if (!planned && !fold) rc = launch_prep(p, st);
  if (rc != PNCE_OK) return rc;
  int ctas_per_image = 0;
  for (int l = 0; l < p.n_layers; ++l) ctas_per_image += p.L[l].Ppad / 128;
  // Chunking is OFF by default: on B200 the 14-image chunks that fill the SMs once make the gather
  // pay ~30% wave quantisation and the overlap does not win it back (measured: 0.70 ms vs 0.50 ms
  // forward at B=64).  Kept behind the debug knob for larger batches.
  int nchunk = (g_dbg.fwd_chunks > 1 && !p.mb) ? g_dbg.fwd_chunks : 1;   // an mb item needs the keys of every image
  if (nchunk > 16) nchunk = 16;
  if (nchunk > p.B) nchunk = p.B;
  int per = (p.B + nchunk - 1) / nchunk;
  nchunk = (p.B + per - 1) / per;
  p.total_ctas = (unsigned)(p.B * ctas_per_image);
  if (nchunk == 1) {
    p.b0 = 0; p.bn = p.B;
    rc = launch_gather_tc(p, st, fold);
    if (rc != PNCE_OK) return rc;
    if (g_dbg.post_gather_event) PNCE_CUDA(cudaEventRecord(g_dbg.post_gather_event, st));
    for (int r = 0; r < g_dbg.loss_repeat; ++r) {              // experiment: warm launches in front of the real one
      rc = launch_loss_tc(p, st);
      if (rc != PNCE_OK) return rc;
    }
    return launch_loss_tc(p, st);
  }
  AuxStreams* ax = nullptr;
  rc = aux_streams(&ax);
  if (rc != PNCE_OK) return rc;
  for (int c = 0; c < nchunk; ++c) {
    p.b0 = c * per;
    p.bn = (p.b0 + per <= p.B) ? per : p.B - p.b0;
    rc = launch_gather_tc(p, st);
    if (rc != PNCE_OK) return rc;
    PNCE_CUDA(cudaEventRecord(ax->ev[c], st));
    PNCE_CUDA(cudaStreamWaitEvent(ax->aux, ax->ev[c], 0));
    rc = launch_loss_tc(p, ax->aux, false);
    if (rc != PNCE_OK) return rc;
  }
  PNCE_CUDA(cudaEventRecord(ax->join, ax->aux));
  PNCE_CUDA(cudaStreamWaitEvent(st, ax->join, 0));
  return PNCE_OK;
}

static int launch_dense_nhwc(const Params& p, cudaStream_t st) {
  const size_t es = dtype_size(p.dtype);
  DenseNhwcMap f;
  memset(&f, 0, sizeof(f));
  bool vec = true;
  long long tot = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    const size_t rowbytes = (size_t)p.L[l].C * es;
    if (rowbytes > kFlatBytes) return PNCE_ERR_UNSUPPORTED;
    f.start[l] = tot;
    f.tpos[l] = (int)(kFlatBytes / rowbytes);
    f.tiles[l] = (p.L[l].HW + f.tpos[l] - 1) / f.tpos[l];
    if ((rowbytes % 16 != 0) || (reinterpret_cast<uintptr_t>(p.L[l].dtgt) & 15u)) vec = false;
    tot += (long long)p.B * f.tiles[l];
  }
  f.start[p.n_layers] = tot;
  if (tot > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  const unsigned grid = (unsigned)tot;
  bool two = vec && !(g_dbg.dense_flags & 32);               // experiment bit 32: the one-launch kernel
  for (int l = 0; l < p.n_layers && two; ++l) two = (p.L[l].C % 4) == 0 && p.L[l].C <= 256;
  if (two) {
    // bare zero fill of every map, then the sampled rows (nhwc.cuh)
    FillMap fm;
    ScatterMap sm;
    memset(&fm, 0, sizeof(fm));
    memset(&sm, 0, sizeof(sm));
    long long tiles = 0, items = 0;
    fm.n = p.n_layers;
    for (int l = 0; l < p.n_layers; ++l) {
      fm.start[l] = tiles;
      fm.bytes[l] = (unsigned long long)p.B * p.L[l].HW * p.L[l].C * es;
      fm.base[l] = p.L[l].dtgt;
      tiles += (long long)((fm.bytes[l] + kFlatBytes - 1) / kFlatBytes);
      sm.start[l] = items;
      items += (long long)p.B * p.L[l].P;
    }
    fm.start[p.n_layers] = tiles;
    sm.start[p.n_layers] = items;
    if (tiles > 0x7fffffffLL || items > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
    launch_k<0>(k_fill_zero, (unsigned)tiles, 128, 0, st, fm);
    PNCE_CUDA(cudaGetLastError());
    const unsigned sgrid = (unsigned)((items + 7) / 8);
    if (p.dtype == PNCE_F32) launch_k<0>(k_scatter_nhwc<float>, sgrid, 256, 0, st, p, sm);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_scatter_nhwc<__half>, sgrid, 256, 0, st, p, sm);
    else launch_k<0>(k_scatter_nhwc<__nv_bfloat16>, sgrid, 256, 0, st, p, sm);
    PNCE_CUDA(cudaGetLastError());
    return PNCE_OK;
  }
  if (vec) {
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_nhwc<float, true>, grid, 128, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_nhwc<__half, true>, grid, 128, 0, st, p, f);
    else launch_k<0>(k_dense_nhwc<__nv_bfloat16, true>, grid, 128, 0, st, p, f);
  } else {
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_nhwc<float, false>, grid, 128, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_nhwc<__half, false>, grid, 128, 0, st, p, f);
    else launch_k<0>(k_dense_nhwc<__nv_bfloat16, false>, grid, 128, 0, st, p, f);
  }
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int launch_dense(const Params& p, cudaStream_t st) {
  if (p.nhwc) return launch_dense_nhwc(p, st);
  const size_t es = dtype_size(p.dtype);
  // default: one small CTA per 8 KB tile, in address order
  DenseFlatMap f;
  memset(&f, 0, sizeof(f));
  bool vec = true;
  long long tot = 0;
  const int tp = kFlatBytes / (int)es;
  for (int l = 0; l < p.n_layers; ++l) {
    f.start[l] = tot;
    f.tiles[l] = (p.L[l].HW + tp - 1) / tp;
    // 128-bit copy-out needs every row start and every tile to be 16-byte aligned
    if ((((size_t)p.L[l].HW * es) % 16 != 0) || (reinterpret_cast<uintptr_t>(p.L[l].dtgt) & 15u)) vec = false;
    tot += (long long)p.B * p.L[l].C * f.tiles[l];
  }
  f.start[p.n_layers] = tot;
  f.flags = g_dbg.dense_flags;
  if (tot > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  const unsigned grid = (unsigned)tot;
  if (vec && (g_dbg.dense_flags & 2)) {                      // experiment: store-first variant
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_direct<float, 128>, grid, 128, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_direct<__half, 128>, grid, 128, 0, st, p, f);
    else launch_k<0>(k_dense_direct<__nv_bfloat16, 128>, grid, 128, 0, st, p, f);
  } else if (vec && (g_dbg.dense_flags & 4)) {               // experiment: 64-thread CTAs (more tiles in flight per SM)
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_flat<float, 64, true>, grid, 64, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_flat<__half, 64, true>, grid, 64, 0, st, p, f);
    else launch_k<0>(k_dense_flat<__nv_bfloat16, 64, true>, grid, 64, 0, st, p, f);
  } else if (vec) {
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_flat<float, 128, true>, grid, 128, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_flat<__half, 128, true>, grid, 128, 0, st, p, f);
    else launch_k<0>(k_dense_flat<__nv_bfloat16, 128, true>, grid, 128, 0, st, p, f);
  } else {
    if (p.dtype == PNCE_F32) launch_k<0>(k_dense_flat<float, 128, false>, grid, 128, 0, st, p, f);
    else if (p.dtype == PNCE_F16) launch_k<0>(k_dense_flat<__half, 128, false>, grid, 128, 0, st, p, f);
    else launch_k<0>(k_dense_flat<__nv_bfloat16, 128, false>, grid, 128, 0, st, p, f);
  }
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int check_alignment(const pnce_layer_t* layers, int n_layers, int dtype, bool need_dtgt) {
  const uintptr_t mask = dtype_size(dtype) - 1;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    if (a.ids == nullptr || (reinterpret_cast<uintptr_t>(a.ids) & 7u)) return PNCE_ERR_ARG;
    if (!need_dtgt) {
      if (a.src == nullptr || a.tgt == nullptr) return PNCE_ERR_ARG;
      if ((reinterpret_cast<uintptr_t>(a.src) & mask) || (reinterpret_cast<uintptr_t>(a.tgt) & mask))
        return PNCE_ERR_ALIGN;
    } else {
      if (a.dtgt == nullptr) return PNCE_ERR_ARG;
      if (reinterpret_cast<uintptr_t>(a.dtgt) & mask) return PNCE_ERR_ALIGN;
    }
  }
  return PNCE_OK;
}

}  // namespace pnce

using namespace pnce;

extern "C" {

int pnce_abi_version(void) { return PNCE_ABI_VERSION; }

const char* pnce_status_string(int s) {
  switch (s) {
    case PNCE_OK: return "ok";
    case PNCE_ERR_ARG: return "invalid argument";
    case PNCE_ERR_UNSUPPORTED: return "shape outside compiled limits";
    case PNCE_ERR_WORKSPACE: return "workspace too small or misaligned";
    case PNCE_ERR_CUDA: return "CUDA runtime error";
    case PNCE_ERR_ALIGN: return "tensor pointer not element-aligned";
    default: return "unknown status";
  }
}

const char* pnce_last_cuda_error(void) { return g_cuda_err; }

#ifdef PNCE_EXPERIMENTS
// Experiment hooks (libpnce_exp.so only; not part of pnce.h).
int pnce_debug_set(int key, long long value) {
  switch (key) {
    case 1: g_dbg.dense_flags = (int)value; break;
    case 3: g_dbg.trace = reinterpret_cast<long long*>(value); break;
    case 5: g_dbg.fwd_chunks = (int)value; break;
    case 6: g_dbg.no_persist = (int)value; break;
    case 7: g_dbg.persist_ctas = (int)value; break;
    case 8: g_gather_in_layer_order = (int)value; break;
    case 10: g_dbg.post_gather_event = reinterpret_cast<cudaEvent_t>(value); break;
    case 11: g_dbg.loss_rot = value; break;
    case 13: g_dbg.loss_repeat = (int)value; break;
    case 14: g_dbg.gemm_dbg = (int)value; break;
    case 9: { int v = (int)value; PNCE_CUDA(cudaMemcpyToSymbol(g_dx_evict_last, &v, sizeof(int))); break; }
    default: return PNCE_ERR_ARG;
  }
  return PNCE_OK;
}
// Experiment: occupy `n_sms` SMs (one CTA with 227 KB of shared memory each) until *stop != 0 (bounded, ~40 ms):
// what do the other kernels lose when a persistent kernel owns part of the GPU?
__global__ void k_debug_blocker(volatile int* stop, int* resident) {
  pdl_enter();
  extern __shared__ unsigned char bs[];
  if (threadIdx.x == 0) atomicAdd(resident, 1);
  const long long t0 = clock64();
  while (clock64() - t0 < 80000000ll) {
    if (*stop != 0) break;
    __nanosleep(10000);
  }
  if (bs[0] == 77 && *stop == 12345) *resident = -1;
}
int pnce_debug_block_sms(int n_sms, int* stop_and_resident, void* stream) {
  PNCE_CUDA(cudaFuncSetAttribute(k_debug_blocker, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
  k_debug_blocker<<<n_sms, 1, 226 * 1024, static_cast<cudaStream_t>(stream)>>>(stop_and_resident, stop_and_resident + 1);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}
// Experiment (scratch/exp31.py): zero fill by 128-thread CTAs without shared memory -- can it run beside k_loss_tc_p?
// ctas > 0: persistent grid-stride CTAs; ctas == 0: one CTA per 8 KB, in address order.
__global__ void __launch_bounds__(128) k_debug_fill(float4* __restrict__ p, long long n16, int persistent) {
  pdl_enter();
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  if (persistent) {
    for (long long i = (long long)blockIdx.x * 128 + threadIdx.x; i < n16; i += (long long)gridDim.x * 128) p[i] = z;
  } else {
    const long long base = (long long)blockIdx.x * 512;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long i = base + k * 128 + threadIdx.x;
      if (i < n16) p[i] = z;
    }
  }
}
int pnce_debug_fill(void* ptr, long long bytes, int ctas, void* stream) {
  PNCE_CUDA(cudaFuncSetAttribute(k_debug_fill, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  const long long n16 = bytes / 16;
  const unsigned grid = ctas > 0 ? (unsigned)ctas : (unsigned)((n16 + 511) / 512);
  k_debug_fill<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<float4*>(ptr), n16, ctas > 0);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}
// device-wide L2 fetch granularity hint, 32/64/128 bytes
int pnce_debug_set_l2_fetch_granularity(int bytes) {
  PNCE_CUDA(cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes));
  size_t v = 0;
  PNCE_CUDA(cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity));
  return (int)v;
}
#endif  // PNCE_EXPERIMENTS

int pnce_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  size_t need = carve_fused(layers, n_layers, batch, false, false, nullptr, nullptr);
  if (tc_shapes_ok(layers, n_layers)) {
    const size_t t = carve_fused(layers, n_layers, batch, true, true, nullptr, nullptr);
    if (t > need) need = t;
  }
  *bytes = need;
  return PNCE_OK;
}

static int fwd_impl(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
                    int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes, float* loss_out,
                    int* nonfinite, void* stream, const unsigned long long* rng = nullptr, int layout = PNCE_LAYOUT_NCHW,
                    bool mb = false) {
  int rc = check_layers(layers, n_layers, batch);
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (rc != PNCE_OK) return rc;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16 || loss_out == nullptr || !(temperature > 0.f)) return PNCE_ERR_ARG;
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  rc = check_alignment(layers, n_layers, dtype, false);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  // the tcgen05 kernel covers P <= 1024, C <= 256 (every CUT layer up to the 512^2 stress config); other shapes take the
  // fp32 CUDA-core kernel -- both are device paths of this library, neither is a fallback off the GPU
  const bool tc = math_mode != PNCE_MATH_SIMT_F32 && tc_shapes_ok(layers, n_layers);
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  if (mb && (!tc || !mb_shapes_ok(layers, n_layers, batch))) return PNCE_ERR_UNSUPPORTED;
  if (plan != nullptr) {
    if (!tc) return PNCE_ERR_UNSUPPORTED;                      // planned ids: tensor-core path only
    if ((reinterpret_cast<uintptr_t>(plan) & 255u) || carve_plan(layers, n_layers, nullptr, nullptr) > plan_bytes)
      return PNCE_ERR_WORKSPACE;
  }
  Params p;
  if (carve_fused(layers, n_layers, batch, tc, x3, ws, &p, plan) > ws_bytes) return PNCE_ERR_WORKSPACE;
  p.dtype = dtype;
  p.math = tc ? math_mode : PNCE_MATH_SIMT_F32;
  p.tau = temperature;
  p.loss_out = loss_out;
  p.nonfinite = nonfinite;
  p.trace = g_dbg.trace;
  p.b0 = 0; p.bn = batch;
  p.mb = mb ? 1 : 0;
  if (layout == PNCE_LAYOUT_NHWC) {
    if (!tc) return PNCE_ERR_UNSUPPORTED;                      // channels-last maps: tensor-core path only
    p.nhwc = 1;
  }
  if (rng != nullptr) {
    if (!tc || plan != nullptr) return PNCE_ERR_UNSUPPORTED;   // the draw rides on k_prep (tensor-core path, unplanned)
    p.rng_draw = 1; p.rng_seed = rng[0]; p.rng_offset = rng[1];
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (tc) return forward_tc(p, st, plan != nullptr);
  rc = launch_gather(p, n_layers, st);
  if (rc != PNCE_OK) return rc;
  return launch_loss_simt(p, st);
}

int pnce_fwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
             int math_mode, void* ws, size_t ws_bytes, float* loss_out, int* nonfinite, void* stream) {
  return fwd_impl(layers, n_layers, batch, dtype, temperature, math_mode, ws, ws_bytes, nullptr, 0, loss_out,
                  nonfinite, stream);
}

int pnce_fwd_draw(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
                  int math_mode, void* ws, size_t ws_bytes, unsigned long long philox_seed,
                  unsigned long long philox_offset, float* loss_out, int* nonfinite, void* stream) {
  const unsigned long long rng[2] = {philox_seed, philox_offset};
  return fwd_impl(layers, n_layers, batch, dtype, temperature, math_mode, ws, ws_bytes, nullptr, 0, loss_out,
                  nonfinite, stream, rng);
}

int pnce_fwd_planned(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
                     int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes, float* loss_out,
                     int* nonfinite, void* stream) {
  if (plan == nullptr) return PNCE_ERR_ARG;
  return fwd_impl(layers, n_layers, batch, dtype, temperature, math_mode, ws, ws_bytes, plan, plan_bytes,
                  loss_out, nonfinite, stream);
}

int pnce_plan_bytes(const pnce_layer_t* layers, int n_layers, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, 1);
  if (rc != PNCE_OK) return rc;
  *bytes = carve_plan(layers, n_layers, nullptr, nullptr);
  return PNCE_OK;
}

static int plan_ids_impl(const pnce_layer_t* layers, int n_layers, void* plan, size_t plan_bytes, void* stream,
                         const unsigned long long* rng) {
  int rc = check_layers(layers, n_layers, 1);
  if (rc != PNCE_OK) return rc;
  if (plan == nullptr || (reinterpret_cast<uintptr_t>(plan) & 255u)) return PNCE_ERR_WORKSPACE;
  if (carve_plan(layers, n_layers, nullptr, nullptr) > plan_bytes) return PNCE_ERR_WORKSPACE;
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n_layers;
  p.B = 1;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    if (a.ids == nullptr || (reinterpret_cast<uintptr_t>(a.ids) & 7u)) return PNCE_ERR_ARG;
    LayerDev& L = p.L[l];
    L.ids = reinterpret_cast<const long long*>(a.ids);
    L.C = a.C; L.HW = a.H * a.W; L.P = a.P;
  }
  carve_plan(layers, n_layers, plan, &p);
  if (rng != nullptr) { p.rng_draw = 1; p.rng_seed = rng[0]; p.rng_offset = rng[1]; }
  return launch_prep(p, static_cast<cudaStream_t>(stream));    // counter == nullptr: nothing else is touched
}

int pnce_plan_ids(const pnce_layer_t* layers, int n_layers, void* plan, size_t plan_bytes, void* stream) {
  return plan_ids_impl(layers, n_layers, plan, plan_bytes, stream, nullptr);
}

int pnce_plan_ids_draw(const pnce_layer_t* layers, int n_layers, unsigned long long philox_seed,
                       unsigned long long philox_offset, void* plan, size_t plan_bytes, void* stream) {
  const unsigned long long rng[2] = {philox_seed, philox_offset};
  return plan_ids_impl(layers, n_layers, plan, plan_bytes, stream, rng);
}

// The draw alone (no sort): for callers that only need the ids (PatchSampleF with patch_ids=None).
__global__ void __launch_bounds__(kThreads) k_draw_ids(const __grid_constant__ Params p) {
  pdl_enter();
  const LayerDev& L = p.L[blockIdx.x];
  const unsigned long long off = p.rng_offset + 4ull * blockIdx.x;
  for (int i = threadIdx.x; i < L.P; i += kThreads) {
    curandStatePhilox4_32_10_t st;
    curand_init(p.rng_seed, (unsigned long long)i, off, &st);
    const uint4 r = curand4(&st);
    const_cast<long long*>(L.ids)[i] = (long long)(r.x % (unsigned)L.HW);
  }
}

int pnce_draw_ids(const pnce_layer_t* layers, int n_layers, unsigned long long philox_seed,
                  unsigned long long philox_offset, void* stream) {
  int rc = check_layers(layers, n_layers, 1);
  if (rc != PNCE_OK) return rc;
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n_layers;
  p.rng_draw = 1; p.rng_seed = philox_seed; p.rng_offset = philox_offset;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    if (a.ids == nullptr || (reinterpret_cast<uintptr_t>(a.ids) & 7u)) return PNCE_ERR_ARG;
    p.L[l].ids = reinterpret_cast<const long long*>(a.ids);
    p.L[l].HW = a.H * a.W; p.L[l].P = a.P;
  }
  launch_k(k_draw_ids, (unsigned)n_layers, kThreads, 0, static_cast<cudaStream_t>(stream), p);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int bwd_impl(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int math_mode, void* ws,
                    size_t ws_bytes, void* plan, size_t plan_bytes, const float* grad_out, void* stream,
                    int layout = PNCE_LAYOUT_NCHW) {
  int rc = check_layers(layers, n_layers, batch);
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (rc != PNCE_OK) return rc;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  rc = check_alignment(layers, n_layers, dtype, true);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  const bool tc = math_mode != PNCE_MATH_SIMT_F32 && tc_shapes_ok(layers, n_layers);
  if (plan != nullptr && (!tc || carve_plan(layers, n_layers, nullptr, nullptr) > plan_bytes)) return PNCE_ERR_WORKSPACE;
  Params p;
  if (carve_fused(layers, n_layers, batch, tc, math_mode == PNCE_MATH_TC_BF16X3, ws, &p, plan) > ws_bytes)
    return PNCE_ERR_WORKSPACE;
  p.dtype = dtype;
  p.grad_out = grad_out;
  if (layout == PNCE_LAYOUT_NHWC) {
    if (!tc) return PNCE_ERR_UNSUPPORTED;
    p.nhwc = 1;
  }
  return launch_dense(p, static_cast<cudaStream_t>(stream));
}

int pnce_fwd_ex(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, float temperature,
                int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes,
                const unsigned long long* philox, float* loss_out, int* nonfinite, void* stream) {
  return fwd_impl(layers, n_layers, batch, dtype, temperature, math_mode, ws, ws_bytes, plan, plan_bytes, loss_out,
                  nonfinite, stream, philox, layout);
}

int pnce_bwd_ex(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, int math_mode, void* ws,
                size_t ws_bytes, void* plan, size_t plan_bytes, const float* grad_out, void* stream) {
  return bwd_impl(layers, n_layers, batch, dtype, math_mode, ws, ws_bytes, plan, plan_bytes, grad_out, stream, layout);
}

int pnce_bwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int math_mode, void* ws,
             size_t ws_bytes, const float* grad_out, void* stream) {
  return bwd_impl(layers, n_layers, batch, dtype, math_mode, ws, ws_bytes, nullptr, 0, grad_out, stream);
}

int pnce_bwd_planned(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int math_mode, void* ws,
                     size_t ws_bytes, void* plan, size_t plan_bytes, const float* grad_out, void* stream) {
  if (plan == nullptr) return PNCE_ERR_ARG;
  return bwd_impl(layers, n_layers, batch, dtype, math_mode, ws, ws_bytes, plan, plan_bytes, grad_out, stream);
}

// ---- minibatch negatives (nce_includes_all_negatives_from_minibatch) ----------------------------------------------
int pnce_mb_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!mb_shapes_ok(layers, n_layers, batch)) return PNCE_ERR_UNSUPPORTED;
  *bytes = carve_fused(layers, n_layers, batch, true, true, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_mb_fwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, float temperature,
                int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes,
                const unsigned long long* philox, float* loss_out, int* nonfinite, void* stream) {
  if (math_mode == PNCE_MATH_SIMT_F32) return PNCE_ERR_UNSUPPORTED;
  const int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!mb_shapes_ok(layers, n_layers, batch)) return PNCE_ERR_UNSUPPORTED;
  return fwd_impl(layers, n_layers, batch, dtype, temperature, math_mode, ws, ws_bytes, plan, plan_bytes, loss_out,
                  nonfinite, stream, philox, layout, true);
}

// ---- global negatives: minibatch negatives over the shards of every rank (configs/train_gan_cutpp.yaml:80,
//      patchnce_cut.py:42-110 on the group of world * batch_local * P rows) ---------------------------------------------
// Workspace: the prefix of pnce_mb_workspace_bytes(batch_local) (query blobs, id tables, gradient rows -- what
// pnce_bwd_ex reads), then `world` slots.  A slot holds one rank's qbad flags and, per layer, its key blobs khi, k2hi,
// kss, klo, k2lo for batch_local images, every piece 256-byte aligned.  The low parts are reserved in both tensor-core
// modes so that the layout does not depend on the math mode.
static size_t carve_mb_slot(const pnce_layer_t* layers, int n_layers, int B, bool x3, void* base, Params* p) {
  Carver cv(base);
  int* flags = cv.take<int>(PNCE_MAX_LAYERS);
  if (p != nullptr) p->qbad = flags;
  for (int l = 0; l < n_layers; ++l) {
    const size_t Ppad = (layers[l].P + 127) / 128 * 128, Cp = (layers[l].C + 31) / 32 * 32, nchunk = Cp / 32;
    const size_t blob = (size_t)B * Ppad * Cp;
    __nv_bfloat16* khi = cv.take<__nv_bfloat16>(blob);
    __nv_bfloat16* k2hi = cv.take<__nv_bfloat16>(blob);
    float* kss = cv.take<float>((size_t)B * nchunk * Ppad);
    __nv_bfloat16* klo = cv.take<__nv_bfloat16>(blob);
    __nv_bfloat16* k2lo = cv.take<__nv_bfloat16>(blob);
    if (p != nullptr) {
      LayerDev& L = p->L[l];
      L.khi = khi; L.k2hi = k2hi; L.kss = kss;
      L.klo = x3 ? klo : nullptr;
      L.k2lo = x3 ? k2lo : nullptr;
    }
  }
  return align_up(cv.off, 256);
}

// Keys call, after this rank's query sums of squares exist: its "a query row is non-finite" flags (k_mb_qbad on p's qss,
// every layer) into `flags`, which live in its slot next to its keys.
static int launch_mb_qbad(const Params& p, int* flags, cudaStream_t st) {
  PNCE_CUDA(cudaMemsetAsync(flags, 0, PNCE_MAX_LAYERS * sizeof(int), st));
  long long most = 1;
  for (int l = 0; l < p.n_layers; ++l) {
    const long long n = (long long)p.B * p.L[l].nchunk * p.L[l].Ppad;
    if ((n + kMbQbadFloats - 1) / kMbQbadFloats > most) most = (n + kMbQbadFloats - 1) / kMbQbadFloats;
  }
  if (most > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  launch_k<2>(k_mb_qbad, dim3((unsigned)most, (unsigned)p.n_layers), kThreads, 0, st, p, flags);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

// Loss call, once p's key blobs and qbad point at slot 0: k_loss_tc_mb_gn steps to slot w by w * kslot, and this rank's
// query images are global images rank * B on.
static void point_at_slots(Params& p, int world, int rank, size_t slot_bytes) {
  p.kworld = world;
  p.kimg0 = rank * p.B;
  p.kslot = slot_bytes;
  int ctas_per_image = 0;
  for (int l = 0; l < p.n_layers; ++l) ctas_per_image += p.L[l].Ppad / 128;
  p.total_ctas = (unsigned)(p.B * ctas_per_image);
}

// The envelope of the global batch and the slot geometry: *prefix, the slots' offset; *slot_bytes, their stride.  No
// CUDA call.
static int mb_shard_geometry(const pnce_layer_t* layers, int n_layers, int batch_local, int world, size_t* prefix,
                             size_t* slot_bytes) {
  const int rc = global_batch_check(world, batch_local, [&](int B) {
    return mb_shapes_ok(layers, n_layers, B) ? PNCE_OK : PNCE_ERR_UNSUPPORTED;
  });
  if (rc != PNCE_OK) return rc;
  *prefix = carve_fused(layers, n_layers, batch_local, true, true, nullptr, nullptr);
  *slot_bytes = carve_mb_slot(layers, n_layers, batch_local, true, nullptr, nullptr);
  return PNCE_OK;
}

// The checks of both shard calls, all before any CUDA call; fills Params with the prefix carve and with slot `slot`'s
// key blobs.  *slot_bytes: the slot stride.
static int mb_shard_params(const pnce_layer_t* layers, int n_layers, int batch_local, int dtype, int layout, int world,
                           int rank, int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes, int slot,
                           Params* p, size_t* slot_bytes) {
  int rc = check_layers(layers, n_layers, batch_local);
  if (rc != PNCE_OK) return rc;
  if (world < 1 || rank < 0 || rank >= world) return PNCE_ERR_ARG;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  if (math_mode == PNCE_MATH_SIMT_F32) return PNCE_ERR_UNSUPPORTED;
  size_t prefix = 0;
  rc = mb_shard_geometry(layers, n_layers, batch_local, world, &prefix, slot_bytes);
  if (rc != PNCE_OK) return rc;
  rc = check_alignment(layers, n_layers, dtype, false);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  if (plan != nullptr &&
      ((reinterpret_cast<uintptr_t>(plan) & 255u) || carve_plan(layers, n_layers, nullptr, nullptr) > plan_bytes))
    return PNCE_ERR_WORKSPACE;
  if (prefix + (size_t)world * *slot_bytes > ws_bytes) return PNCE_ERR_WORKSPACE;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  carve_fused(layers, n_layers, batch_local, true, x3, ws, p, plan);
  carve_mb_slot(layers, n_layers, batch_local, x3, static_cast<unsigned char*>(ws) + prefix + (size_t)slot * *slot_bytes, p);
  p->dtype = dtype;
  p->math = math_mode;
  p->b0 = 0; p->bn = batch_local;
  p->mb = 1;
  p->nhwc = layout == PNCE_LAYOUT_NHWC ? 1 : 0;
  return PNCE_OK;
}

int pnce_mb_shard_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch_local, int world, size_t* bytes,
                                  size_t* slot_offset, size_t* slot_bytes) {
  if (bytes == nullptr || slot_offset == nullptr || slot_bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch_local);
  if (rc != PNCE_OK) return rc;
  if (world < 1) return PNCE_ERR_ARG;
  rc = mb_shard_geometry(layers, n_layers, batch_local, world, slot_offset, slot_bytes);
  if (rc != PNCE_OK) return rc;
  *bytes = *slot_offset + (size_t)world * *slot_bytes;
  return PNCE_OK;
}

int pnce_mb_shard_keys(const pnce_layer_t* layers, int n_layers, int batch_local, int dtype, int layout, int world,
                       int rank, int math_mode, void* ws, size_t ws_bytes, void* plan, size_t plan_bytes,
                       const unsigned long long* philox, void* stream) {
  Params p;
  size_t slot_bytes = 0;
  int rc = mb_shard_params(layers, n_layers, batch_local, dtype, layout, world, rank, math_mode, ws, ws_bytes, plan,
                           plan_bytes, rank, &p, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  if (philox != nullptr) {
    if (plan != nullptr) return PNCE_ERR_UNSUPPORTED;          // the draw rides on the id prep (unplanned)
    p.rng_draw = 1; p.rng_seed = philox[0]; p.rng_offset = philox[1];
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // id prep (unless planned) and the gather: keys straight into slot `rank`, queries into the prefix
  const bool fold = plan == nullptr && gather_tc_folds(p);
  if (plan == nullptr && !fold) rc = launch_prep(p, st);
  if (rc != PNCE_OK) return rc;
  rc = launch_gather_tc(p, st, fold);
  if (rc != PNCE_OK) return rc;
  return launch_mb_qbad(p, const_cast<int*>(p.qbad), st);
}

int pnce_mb_shard_loss(const pnce_layer_t* layers, int n_layers, int batch_local, int dtype, int layout, int world,
                       int rank, float temperature, int math_mode, void* ws, size_t ws_bytes, void* plan,
                       size_t plan_bytes, float* loss_out, int* nonfinite, void* stream) {
  Params p;
  size_t slot_bytes = 0;
  int rc = mb_shard_params(layers, n_layers, batch_local, dtype, layout, world, rank, math_mode, ws, ws_bytes, plan,
                           plan_bytes, 0, &p, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  if (loss_out == nullptr || !(temperature > 0.f)) return PNCE_ERR_ARG;
  p.tau = temperature;
  p.loss_out = loss_out;
  p.nonfinite = nonfinite;
  p.trace = g_dbg.trace;
  point_at_slots(p, world, rank, slot_bytes);
  return launch_loss_tc(p, static_cast<cudaStream_t>(stream));
}

// ---- module-split API ------------------------------------------------------------------------

int pnce_sample_fwd(const void* feat, int dtype, int batch, int C, int H, int W, const int64_t* ids,
                    int P, float* rows_out, float* inv_out, void* stream) {
  pnce_layer_t a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.H = H; a.W = W; a.P = P;
  int rc = check_layers(&a, 1, batch);
  if (rc != PNCE_OK) return rc;
  if (feat == nullptr || ids == nullptr || rows_out == nullptr || dtype < PNCE_F32 || dtype > PNCE_BF16)
    return PNCE_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(feat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = 1; p.B = batch; p.dtype = dtype;
  LayerDev& L = p.L[0];
  L.tgt = feat;
  L.ids = reinterpret_cast<const long long*>(ids);
  L.C = C; L.HW = H * W; L.P = P;
  L.nwords = (L.HW + 31) / 32;
  L.ntiles = (P + kRowTile - 1) / kRowTile;
  L.qn = rows_out;
  L.qinv = inv_out;
  p.side0 = 1;                       // only the "tgt" side exists here
  p.raw = (inv_out == nullptr) ? 1 : 0;
  return launch_gather(p, 0, static_cast<cudaStream_t>(stream));
}

static size_t carve_sample_bwd(int B, int C, int H, int W, int P, void* ws, LayerDev* out) {
  Carver cv(ws);
  LayerDev L;
  memset(&L, 0, sizeof(L));
  L.C = C; L.HW = H * W; L.P = P;
  L.nwords = (L.HW + 31) / 32;
  L.ntiles = (P + kRowTile - 1) / kRowTile;
  L.sid = cv.take<int>(P);
  L.perm = cv.take<int>(P);
  L.rank = cv.take<int>(P);
  L.cslot = cv.take<int>((size_t)(L.HW + kTilePos - 1) / kTilePos + 1);
  L.dxpitch = P;
  L.dxT = cv.take<float>((size_t)B * P * C);
  if (out) *out = L;
  return align_up(cv.off, 256);
}

int pnce_sample_bwd_workspace_bytes(int batch, int C, int H, int W, int P, size_t* bytes) {
  pnce_layer_t a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.H = H; a.W = W; a.P = P;
  int rc = check_layers(&a, 1, batch);
  if (rc != PNCE_OK) return rc;
  if (bytes == nullptr) return PNCE_ERR_ARG;
  *bytes = carve_sample_bwd(batch, C, H, W, P, nullptr, nullptr);
  return PNCE_OK;
}

// One-CTA launch of the id prep alone (module-split backward has no gather to ride on).
__global__ void __launch_bounds__(kThreads) k_prep_only(const __grid_constant__ Params p) {
  pdl_enter();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  int N2 = 1;
  while (N2 < p.L[0].P) N2 <<= 1;
  prep_layer(p.L[0], keys);
}

int pnce_sample_bwd(const float* drows, const float* rows, const float* inv, int dtype, int batch,
                    int C, int H, int W, const int64_t* ids, int P, void* ws, size_t ws_bytes,
                    void* dfeat, void* stream) {
  pnce_layer_t a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.H = H; a.W = W; a.P = P;
  int rc = check_layers(&a, 1, batch);
  if (rc != PNCE_OK) return rc;
  if (!drows || !ids || !dfeat || dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if ((rows == nullptr) != (inv == nullptr)) return PNCE_ERR_ARG;       // both NULL = raw rows (no normalisation)
  if (reinterpret_cast<uintptr_t>(dfeat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  Params p;
  memset(&p, 0, sizeof(p));
  if (carve_sample_bwd(batch, C, H, W, P, ws, &p.L[0]) > ws_bytes) return PNCE_ERR_WORKSPACE;
  p.n_layers = 1; p.B = batch; p.dtype = dtype;
  LayerDev& L = p.L[0];
  L.ids = reinterpret_cast<const long long*>(ids);
  L.qinv = const_cast<float*>(inv);
  L.dtgt = dfeat;
  p.raw = (rows == nullptr) ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int n2 = 1;
  while (n2 < P) n2 <<= 1;
  const size_t prep_smem = (size_t)n2 * 8 + 64;
  launch_k(k_prep_only, 1, kThreads, prep_smem, st, p);
  PNCE_CUDA(cudaGetLastError());
  const size_t smem = (size_t)kRowTile * (C + 1) * sizeof(float);
  rc = set_smem(k_rows_normbwd, smem);
  if (rc != PNCE_OK) return rc;
  launch_k(k_rows_normbwd, (unsigned)(batch * L.ntiles), kThreads, smem, st, p, drows, rows, 0);
  PNCE_CUDA(cudaGetLastError());
  return launch_dense(p, st);
}

// ---- all layers of a PatchSampleF call in one go -------------------------------------------------
static int check_samples(const pnce_sample_t* sm, int n, int batch, int dtype) {
  if (sm == nullptr || n < 1 || batch < 1 || dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (n > PNCE_MAX_LAYERS) return PNCE_ERR_UNSUPPORTED;
  for (int l = 0; l < n; ++l) {
    pnce_layer_t a;
    memset(&a, 0, sizeof(a));
    a.C = sm[l].C; a.H = sm[l].H; a.W = sm[l].W; a.P = sm[l].P;
    int rc = check_layers(&a, 1, batch);
    if (rc != PNCE_OK) return rc;
    if (sm[l].ids == nullptr) return PNCE_ERR_ARG;
  }
  return PNCE_OK;
}

int pnce_sample_multi_fwd(const pnce_sample_t* sm, int n, int batch, int dtype, void* stream) {
  int rc = check_samples(sm, n, batch, dtype);
  if (rc != PNCE_OK) return rc;
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n; p.B = batch; p.dtype = dtype;
  p.side0 = 1;                       // only the "tgt" side exists here
  p.raw = (sm[0].inv == nullptr) ? 1 : 0;
  for (int l = 0; l < n; ++l) {
    if (sm[l].feat == nullptr || sm[l].rows == nullptr) return PNCE_ERR_ARG;
    if ((sm[l].inv == nullptr) != (p.raw != 0)) return PNCE_ERR_ARG;       // raw or normalised, for all layers alike
    if (reinterpret_cast<uintptr_t>(sm[l].feat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
    LayerDev& L = p.L[l];
    L.tgt = sm[l].feat;
    L.ids = reinterpret_cast<const long long*>(sm[l].ids);
    L.C = sm[l].C; L.HW = sm[l].H * sm[l].W; L.P = sm[l].P;
    L.nwords = (L.HW + 31) / 32;
    L.ntiles = (L.P + kRowTile - 1) / kRowTile;
    L.qn = sm[l].rows;
    L.qinv = sm[l].inv;
  }
  return launch_gather(p, 0, static_cast<cudaStream_t>(stream));
}

static size_t carve_sample_multi_bwd(const pnce_sample_t* sm, int n, int B, void* ws, Params* out) {
  Carver cv(ws);
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n; p.B = B;
  for (int l = 0; l < n; ++l) {
    LayerDev& L = p.L[l];
    L.C = sm[l].C; L.HW = sm[l].H * sm[l].W; L.P = sm[l].P;
    L.nwords = (L.HW + 31) / 32;
    L.ntiles = (L.P + kRowTile - 1) / kRowTile;
    L.sid = cv.take<int>(L.P);
    L.perm = cv.take<int>(L.P);
    L.rank = cv.take<int>(L.P);
    L.cslot = cv.take<int>((size_t)(L.HW + kTilePos - 1) / kTilePos + 1);
    L.dxpitch = L.P;
    L.dxT = cv.take<float>((size_t)B * L.P * L.C);
  }
  if (out) *out = p;
  return align_up(cv.off, 256);
}

int pnce_sample_multi_bwd_workspace_bytes(const pnce_sample_t* sm, int n, int batch, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_samples(sm, n, batch, PNCE_F32);
  if (rc != PNCE_OK) return rc;
  *bytes = carve_sample_multi_bwd(sm, n, batch, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_sample_multi_bwd(const pnce_sample_t* sm, int n, int batch, int dtype, void* ws, size_t ws_bytes,
                          void* stream) {
  int rc = check_samples(sm, n, batch, dtype);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  Params p;
  if (carve_sample_multi_bwd(sm, n, batch, ws, &p) > ws_bytes) return PNCE_ERR_WORKSPACE;
  p.dtype = dtype;
  p.raw = (sm[0].rows == nullptr) ? 1 : 0;
  size_t smem = 0;
  for (int l = 0; l < n; ++l) {
    if (sm[l].drows == nullptr || sm[l].dfeat == nullptr) return PNCE_ERR_ARG;
    if ((sm[l].rows == nullptr) != (sm[l].inv == nullptr) || (sm[l].rows == nullptr) != (p.raw != 0)) return PNCE_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(sm[l].dfeat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
    LayerDev& L = p.L[l];
    L.ids = reinterpret_cast<const long long*>(sm[l].ids);
    L.qinv = sm[l].inv;
    L.dtgt = sm[l].dfeat;
    const size_t s = (size_t)kRowTile * (L.C + 1) * sizeof(float);
    if (s > smem) smem = s;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = launch_prep(p, st);                                    // one CTA per layer: sorted ids, ranks, tile slot ranges
  if (rc != PNCE_OK) return rc;
  rc = set_smem(k_rows_normbwd, smem);
  if (rc != PNCE_OK) return rc;
  for (int l = 0; l < n; ++l) {
    const LayerDev& L = p.L[l];
    launch_k(k_rows_normbwd, (unsigned)(batch * L.ntiles), kThreads, (size_t)kRowTile * (L.C + 1) * sizeof(float), st, 
        p, sm[l].drows, sm[l].rows, l);
    PNCE_CUDA(cudaGetLastError());
  }
  return launch_dense(p, st);                                 // every layer's dense gradient in one launch
}

static size_t carve_rows_loss(int B, int P, int D, void* ws, Params* out) {
  Carver cv(ws);
  Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = 1; p.B = B;
  p.counter = cv.take<unsigned>(64);
  p.lossimg = cv.take<float>(B);
  p.valid = cv.take<int>(B);
  LayerDev& L = p.L[0];
  L.C = D; L.P = P; L.HW = 1; L.nwords = 1;
  L.ntiles = (P + kRowTile - 1) / kRowTile;
  L.nparts = L.ntiles;
  L.partial = cv.take<float>((size_t)B * L.ntiles);
  if (out) *out = p;
  return align_up(cv.off, 256);
}

// the same problem on the tensor-core kernel (P, D <= 256): operand blobs + per-chunk norm words, for every layer of a
// PatchSampleF output at once (one pack launch + one loss launch)
static bool rows_tc_ok(int P, int D) { return P <= 256 && D <= 256; }
static size_t carve_rows_multi_tc(const pnce_rows_t* rows, int n, int B, bool x3, void* ws, pnce::Params* out) {
  using namespace pnce;
  Carver cv(ws);
  static thread_local Params p;
  memset(&p, 0, sizeof(p));
  p.n_layers = n; p.B = B; p.rows_mode = 1;
  p.counter = cv.take<unsigned>(64);
  p.lossimg = cv.take<float>((size_t)n * B);
  p.valid = cv.take<int>((size_t)n * B);
  for (int l = 0; l < n; ++l) {
    LayerDev& L = p.L[l];
    const int P = rows[l].P, D = rows[l].D;
    L.C = D; L.P = P; L.HW = 1; L.nwords = 1;
    L.ntiles = (P + kRowTile - 1) / kRowTile;
    L.sorted = 1;
    L.Cp = (D + 31) / 32 * 32;
    L.Ppad = (P + 127) / 128 * 128;
    L.nchunk = L.Cp / 32;
    L.nparts = L.Ppad / 128;
    L.dxpitch = L.Ppad;
    const size_t blob = (size_t)B * L.Ppad * L.Cp;
    L.qhi = cv.take<__nv_bfloat16>(blob);
    L.khi = cv.take<__nv_bfloat16>(blob);
    L.k2hi = cv.take<__nv_bfloat16>(blob);
    if (x3) {
      L.qlo = cv.take<__nv_bfloat16>(blob);
      L.klo = cv.take<__nv_bfloat16>(blob);
      L.k2lo = cv.take<__nv_bfloat16>(blob);
    }
    L.qss = cv.take<float>((size_t)B * L.nchunk * L.Ppad);
    L.kss = cv.take<float>((size_t)B * L.nchunk * L.Ppad);
    L.partial = cv.take<float>((size_t)B * 2);
    L.qn = const_cast<float*>(rows[l].q);
    L.kn = const_cast<float*>(rows[l].k);
    L.dq_rows = rows[l].dq;
  }
  if (out) *out = p;
  return align_up(cv.off, 256);
}

// Re-tiles the rows of every layer into operand blobs (k_rows_pack), after the counter reset the loss kernel relies on.
static int launch_rows_pack(const Params& t, cudaStream_t st) {
  PNCE_CUDA(cudaMemsetAsync(t.counter, 0, 2 * sizeof(unsigned), st));
  long long most = 0;
  for (int l = 0; l < t.n_layers; ++l) {
    const long long threads = 2ll * t.B * t.L[l].Ppad * (t.L[l].Cp >> 3);
    if (threads > most) most = threads;
  }
  launch_k(k_rows_pack, dim3((unsigned)((most + kThreads - 1) / kThreads), (unsigned)t.n_layers), kThreads, 0, st, t);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

int pnce_rows_loss_workspace_bytes(int batch, int P, int D, size_t* bytes) {
  if (bytes == nullptr || batch < 1 || P < 1 || D < 1) return PNCE_ERR_ARG;
  if (P > PNCE_MAX_PATCHES || D > PNCE_MAX_CHANNELS) return PNCE_ERR_UNSUPPORTED;
  size_t need = carve_rows_loss(batch, P, D, nullptr, nullptr);
  if (rows_tc_ok(P, D)) {
    const pnce_rows_t row = {nullptr, nullptr, nullptr, P, D};
    const size_t t = carve_rows_multi_tc(&row, 1, batch, true, nullptr, nullptr);
    if (t > need) need = t;
  }
  *bytes = need;
  return PNCE_OK;
}

int pnce_rows_loss_fwd_bwd(const float* q, const float* k, int batch, int P, int D, float temperature,
                           int math_mode, void* ws, size_t ws_bytes, float* loss_out, int* nonfinite,
                           float* dq_out, float* dk_out, void* stream) {
  if (!q || !k || !loss_out || !dq_out || batch < 1 || P < 1 || D < 1 || !(temperature > 0.f)) return PNCE_ERR_ARG;
  if (P > PNCE_MAX_PATCHES || D > PNCE_MAX_CHANNELS) return PNCE_ERR_UNSUPPORTED;
  if (dk_out != nullptr) return PNCE_ERR_UNSUPPORTED;   // feat_k is detached in the reference (:142)
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  cudaStream_t st0 = static_cast<cudaStream_t>(stream);
  if (math_mode != PNCE_MATH_SIMT_F32 && rows_tc_ok(P, D)) {
    // tensor-core modes: re-tile the rows into operand blobs (k_rows_pack), then the tcgen05 loss kernel in
    // rows mode (rows used as given, d loss / d q written row-major).  P or D > 256: CUDA-core kernel below.
    const pnce_rows_t row = {q, k, dq_out, P, D};
    Params t;
    if (carve_rows_multi_tc(&row, 1, batch, math_mode == PNCE_MATH_TC_BF16X3, ws, &t) > ws_bytes)
      return PNCE_ERR_WORKSPACE;
    t.math = math_mode;
    t.tau = temperature;
    t.loss_out = loss_out;
    t.nonfinite = nonfinite;
    t.b0 = 0; t.bn = batch;
    const int rc = launch_rows_pack(t, st0);
    if (rc != PNCE_OK) return rc;
    return launch_loss_tc(t, st0);
  }
  // fp32 CUDA-core kernel on the rows as they are
  Params p;
  if (carve_rows_loss(batch, P, D, ws, &p) > ws_bytes) return PNCE_ERR_WORKSPACE;
  p.tau = temperature;
  p.loss_out = loss_out;
  p.nonfinite = nonfinite;
  LayerDev& L = p.L[0];
  L.qn = const_cast<float*>(q);
  L.kn = const_cast<float*>(k);
  L.dq_rows = dq_out;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PNCE_CUDA(cudaMemsetAsync(p.counter, 0, 2 * sizeof(unsigned), st));
  return launch_loss_simt(p, st);
}

static int check_rows_multi(const pnce_rows_t* rows, int n, int batch) {
  if (rows == nullptr || n < 1 || n > PNCE_MAX_LAYERS || batch < 1) return PNCE_ERR_ARG;
  for (int l = 0; l < n; ++l) {
    if (rows[l].P < 1 || rows[l].D < 1) return PNCE_ERR_ARG;
    if (!rows_tc_ok(rows[l].P, rows[l].D)) return PNCE_ERR_UNSUPPORTED;
  }
  return PNCE_OK;
}

int pnce_rows_loss_multi_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_rows_multi(rows, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  *bytes = carve_rows_multi_tc(rows, n_layers, batch, true, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_rows_loss_multi_fwd_bwd(const pnce_rows_t* rows, int n_layers, int batch, float temperature, int math_mode,
                                 void* ws, size_t ws_bytes, float* loss_out, int* nonfinite, void* stream) {
  using namespace pnce;
  int rc = check_rows_multi(rows, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!loss_out || !(temperature > 0.f)) return PNCE_ERR_ARG;
  if (math_mode != PNCE_MATH_TC_BF16X3 && math_mode != PNCE_MATH_TC_BF16) return PNCE_ERR_UNSUPPORTED;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  for (int l = 0; l < n_layers; ++l)
    if (!rows[l].q || !rows[l].k || !rows[l].dq) return PNCE_ERR_ARG;
  static thread_local Params t;
  if (carve_rows_multi_tc(rows, n_layers, batch, math_mode == PNCE_MATH_TC_BF16X3, ws, &t) > ws_bytes)
    return PNCE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  t.math = math_mode;
  t.tau = temperature;
  t.loss_out = loss_out;
  t.nonfinite = nonfinite;
  t.b0 = 0; t.bn = batch;
  rc = launch_rows_pack(t, st);
  if (rc != PNCE_OK) return rc;
  return launch_loss_tc(t, st);
}

static int check_rows_mb(const pnce_rows_t* rows, int n, int batch) {
  if (rows == nullptr || n < 1 || n > PNCE_MAX_LAYERS || batch < 1) return PNCE_ERR_ARG;
  for (int l = 0; l < n; ++l) {
    if (rows[l].P < 1 || rows[l].D < 1) return PNCE_ERR_ARG;
    if (!rows_tc_ok(rows[l].P, rows[l].D) || !mb_keys_ok(batch, rows[l].P)) return PNCE_ERR_UNSUPPORTED;
  }
  return PNCE_OK;
}

int pnce_rows_mb_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_rows_mb(rows, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  *bytes = carve_rows_multi_tc(rows, n_layers, batch, true, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_rows_mb_fwd_bwd(const pnce_rows_t* rows, int n_layers, int batch, float temperature, int math_mode,
                         void* ws, size_t ws_bytes, float* loss_out, int* nonfinite, void* stream) {
  using namespace pnce;
  int rc = check_rows_mb(rows, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!loss_out || !(temperature > 0.f)) return PNCE_ERR_ARG;
  if (math_mode != PNCE_MATH_TC_BF16X3 && math_mode != PNCE_MATH_TC_BF16) return PNCE_ERR_UNSUPPORTED;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  for (int l = 0; l < n_layers; ++l) {
    if (!rows[l].q || !rows[l].k || !rows[l].dq) return PNCE_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(rows[l].dq) & 31u) return PNCE_ERR_ALIGN;   // 32-byte row stores (k_loss_tc_mb)
  }
  static thread_local Params t;
  if (carve_rows_multi_tc(rows, n_layers, batch, math_mode == PNCE_MATH_TC_BF16X3, ws, &t) > ws_bytes)
    return PNCE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  t.math = math_mode;
  t.tau = temperature;
  t.loss_out = loss_out;
  t.nonfinite = nonfinite;
  t.b0 = 0; t.bn = batch;
  t.mb = 1;
  t.total_ctas = 0;
  for (int l = 0; l < n_layers; ++l) t.total_ctas += (unsigned)(batch * (t.L[l].Ppad / 128));
  rc = launch_rows_pack(t, st);
  if (rc != PNCE_OK) return rc;
  return launch_loss_tc(t, st);
}

// ---- row route with global negatives: minibatch negatives over the row shards of every rank ---------------------------
// Workspace: the prefix pnce_rows_mb_workspace_bytes(batch_local) (carve_rows_multi_tc: counter, per-layer losses, the
// query blobs and sums of squares, the row-loss partials), then `world` slots in the format of pnce_mb_shard_*
// (carve_mb_slot with C = D).  k_rows_pack writes this rank's keys straight into its slot (its key blobs and kss are the
// gather's, one key block per image); carve_rows_multi_tc's own key blobs stay unused in this mode.
//
// The query flags: k_mb_qbad on the prefix's qss.  k_rows_pack writes 1 (chunk 0) and 0 (the others) for a finite row,
// NaN for every chunk of a row holding a NaN / Inf, 0 for padding, so a flag is raised exactly for a row holding a
// non-finite element -- exactly the loss kernel's own row test (badq).  Rows are used as given (norm words 1), so a finite
// row's loss is non-finite only when its exp2 row sum overflows or underflows in the single-pass branch (|q . k| / tau
// beyond ~88 - ln N: rows far from unit norm, DESIGN.md 4.15): the one case where the owning rank guards alone.

// The envelope of the GLOBAL batch (world * batch_local images) and the slot geometry (vl: the layers carve_mb_slot
// reads, C = D); no CUDA call.
static int rows_shard_geometry(const pnce_rows_t* rows, int n, int batch_local, int world, pnce_layer_t* vl,
                               size_t* prefix, size_t* slot_bytes) {
  if (world < 1 || batch_local < 1) return PNCE_ERR_ARG;
  const int rc = global_batch_check(world, batch_local, [&](int B) { return check_rows_mb(rows, n, B); });
  if (rc != PNCE_OK) return rc;
  for (int l = 0; l < n; ++l) {
    memset(&vl[l], 0, sizeof(vl[l]));
    vl[l].C = rows[l].D;
    vl[l].P = rows[l].P;
  }
  *prefix = carve_rows_multi_tc(rows, n, batch_local, true, nullptr, nullptr);
  *slot_bytes = carve_mb_slot(vl, n, batch_local, true, nullptr, nullptr);
  return PNCE_OK;
}

// The checks of both shard calls, all before any CUDA call, then the carve: the prefix into t, and slot `slot`'s key
// blobs and flags over t's.
static int rows_shard_params(const pnce_rows_t* rows, int n, int batch_local, int world, int rank, int math_mode,
                             void* ws, size_t ws_bytes, int slot, Params& t, size_t* slot_bytes) {
  pnce_layer_t vl[PNCE_MAX_LAYERS];
  size_t prefix = 0;
  int rc = rows_shard_geometry(rows, n, batch_local, world, vl, &prefix, slot_bytes);
  if (rc != PNCE_OK) return rc;
  if (rank < 0 || rank >= world) return PNCE_ERR_ARG;
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  if (math_mode == PNCE_MATH_SIMT_F32) return PNCE_ERR_UNSUPPORTED;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  if (prefix + (size_t)world * *slot_bytes > ws_bytes) return PNCE_ERR_WORKSPACE;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  carve_rows_multi_tc(rows, n, batch_local, x3, ws, &t);
  carve_mb_slot(vl, n, batch_local, x3, static_cast<unsigned char*>(ws) + prefix + (size_t)slot * *slot_bytes, &t);
  t.math = math_mode;
  t.b0 = 0; t.bn = batch_local;
  t.mb = 1;
  return PNCE_OK;
}

int pnce_rows_mb_shard_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch_local, int world, size_t* bytes,
                                       size_t* slot_offset, size_t* slot_bytes) {
  if (bytes == nullptr || slot_offset == nullptr || slot_bytes == nullptr) return PNCE_ERR_ARG;
  pnce_layer_t vl[PNCE_MAX_LAYERS];
  const int rc = rows_shard_geometry(rows, n_layers, batch_local, world, vl, slot_offset, slot_bytes);
  if (rc != PNCE_OK) return rc;
  *bytes = *slot_offset + (size_t)world * *slot_bytes;
  return PNCE_OK;
}

int pnce_rows_mb_shard_keys(const pnce_rows_t* rows, int n_layers, int batch_local, int world, int rank, int math_mode,
                            void* ws, size_t ws_bytes, void* stream) {
  static thread_local Params t;
  size_t slot_bytes = 0;
  int rc = rows_shard_params(rows, n_layers, batch_local, world, rank, math_mode, ws, ws_bytes, rank, t, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  for (int l = 0; l < n_layers; ++l)
    if (!rows[l].q || !rows[l].k) return PNCE_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the pack: queries into the prefix, keys straight into slot `rank`; then this rank's query flags next to its keys
  // (see above for why k_mb_qbad is exact here)
  rc = launch_rows_pack(t, st);
  if (rc != PNCE_OK) return rc;
  return launch_mb_qbad(t, const_cast<int*>(t.qbad), st);
}

int pnce_rows_mb_shard_loss(const pnce_rows_t* rows, int n_layers, int batch_local, int world, int rank,
                            float temperature, int math_mode, void* ws, size_t ws_bytes, float* loss_out, int* nonfinite,
                            void* stream) {
  static thread_local Params t;
  size_t slot_bytes = 0;
  // the key blobs and qbad: slot 0 of `world` (point_at_slots)
  int rc = rows_shard_params(rows, n_layers, batch_local, world, rank, math_mode, ws, ws_bytes, 0, t, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  if (loss_out == nullptr || !(temperature > 0.f)) return PNCE_ERR_ARG;
  for (int l = 0; l < n_layers; ++l) {
    if (!rows[l].dq) return PNCE_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(rows[l].dq) & 31u) return PNCE_ERR_ALIGN;   // 32-byte row stores (k_loss_tc_mb_gn)
  }
  t.tau = temperature;
  t.loss_out = loss_out;
  t.nonfinite = nonfinite;
  point_at_slots(t, world, rank, slot_bytes);
  return launch_loss_tc(t, static_cast<cudaStream_t>(stream));
}

// ---- netF head (tcgen05) ---------------------------------------------------------------------

namespace pnce {

struct HeadLayerBufs {
  __nv_bfloat16 *xq[2], *xk[2], *hq[2], *hk[2], *dh[2];     // [0] = hi, [1] = lo
  __nv_bfloat16 *w1[2], *w2[2], *w1t[2], *w2t[2];
  float *pw2, *pb2, *pw1, *pb1;                              // split-K partials
  int slabs;
};
struct HeadPlan {
  Params pg;                   // the real layers: gather of raw patches, dense backward of dX
  Params pl;                   // "virtual" layers seen by k_loss_tc: C = nc, operands = the head's output
  HeadLayerBufs hb[PNCE_MAX_LAYERS];
};

static bool head_shapes_ok(const pnce_layer_t* layers, int n_layers, int nc) {
  if (nc != 128 && nc != 256) return false;
  for (int l = 0; l < n_layers; ++l)
    if (layers[l].P > 1024 || layers[l].C > 256) return false;
  return true;
}

static size_t carve_head(const pnce_layer_t* layers, int n_layers, int B, int nc, bool x3, void* ws, HeadPlan* out) {
  Carver cv(ws);
  HeadPlan* hp = out;
  HeadPlan local;
  if (hp == nullptr) hp = &local;
  memset(hp, 0, sizeof(HeadPlan));
  Params& pg = hp->pg;
  Params& pl = hp->pl;
  pg.n_layers = pl.n_layers = n_layers;
  pg.B = pl.B = B;
  pl.counter = pg.counter = cv.take<unsigned>(64);
  pl.lossimg = cv.take<float>((size_t)n_layers * B);
  pl.valid = cv.take<int>((size_t)n_layers * B);
  const int nparts = x3 ? 2 : 1;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_layer_t& a = layers[l];
    LayerDev& G = pg.L[l];
    LayerDev& V = pl.L[l];
    HeadLayerBufs& hb = hp->hb[l];
    const int Ppad = (a.P + 127) / 128 * 128, Cp = (a.C + 31) / 32 * 32;
    G.src = a.src; G.tgt = a.tgt; G.dtgt = a.dtgt;
    G.ids = reinterpret_cast<const long long*>(a.ids);
    G.C = a.C; G.HW = a.H * a.W; G.P = a.P;
    G.ntiles = (a.P + kRowTile - 1) / kRowTile;
    G.sorted = 1;
    G.Cp = Cp; G.Ppad = Ppad; G.nchunk = Cp / 32; G.nparts = Ppad / 128;
    G.head_src_rows = 1;
    G.sid = cv.take<int>(a.P);
    G.perm = cv.take<int>(a.P);
    G.rank = cv.take<int>(a.P);
    G.cslot = cv.take<int>((size_t)(G.HW + kTilePos - 1) / kTilePos + 1);
    G.dxpitch = Ppad;
    G.dxT = cv.take<float>((size_t)B * a.C * Ppad);
    const size_t xblob = (size_t)B * Ppad * Cp, yblob = (size_t)B * Ppad * nc;
    for (int k = 0; k < nparts; ++k) {
      hb.xq[k] = cv.take<__nv_bfloat16>(xblob);
      hb.xk[k] = cv.take<__nv_bfloat16>(xblob);
      hb.hq[k] = cv.take<__nv_bfloat16>(yblob);
      hb.hk[k] = cv.take<__nv_bfloat16>(yblob);
      hb.w1[k] = cv.take<__nv_bfloat16>((size_t)nc * Cp);
      hb.w1t[k] = cv.take<__nv_bfloat16>((size_t)nc * Cp);
      hb.w2[k] = cv.take<__nv_bfloat16>((size_t)nc * nc);
      hb.w2t[k] = cv.take<__nv_bfloat16>((size_t)nc * nc);
      hb.dh[k] = hb.hk[k];                                   // H of the key side is dead once Y_k exists
    }
    G.qhi = hb.xq[0]; G.qlo = hb.xq[1]; G.khi = hb.xk[0]; G.klo = hb.xk[1];
    // virtual layer: what k_loss_tc sees
    V = G;
    V.src = V.tgt = nullptr; V.dtgt = nullptr;
    V.C = nc; V.Cp = nc; V.nchunk = nc / 32;
    V.head_src_rows = 0;
    V.qhi = cv.take<__nv_bfloat16>(yblob);
    V.khi = cv.take<__nv_bfloat16>(yblob);
    V.k2hi = cv.take<__nv_bfloat16>(yblob);
    V.dyhi = cv.take<__nv_bfloat16>(yblob);
    if (x3) {
      V.qlo = cv.take<__nv_bfloat16>(yblob);
      V.klo = cv.take<__nv_bfloat16>(yblob);
      V.k2lo = cv.take<__nv_bfloat16>(yblob);
      V.dylo = cv.take<__nv_bfloat16>(yblob);
    } else {
      V.qlo = V.klo = V.k2lo = V.dylo = nullptr;
    }
    V.qss = cv.take<float>((size_t)B * (nc / 32) * Ppad);
    V.kss = cv.take<float>((size_t)B * (nc / 32) * Ppad);
    V.qinv = cv.take<float>((size_t)B * a.P);
    V.kinv = cv.take<float>((size_t)B * Ppad);                  // key-blocked loss kernel (P > 256)
    V.partial = cv.take<float>((size_t)B * (Ppad / 128 > 2 ? Ppad / 128 : 2));
    V.dxT = nullptr;
    const int tiles = B * (Ppad / 128);
    hb.slabs = tiles < 8 ? tiles : 8;
    hb.pw2 = cv.take<float>((size_t)hb.slabs * nc * nc);
    hb.pb2 = cv.take<float>((size_t)hb.slabs * nc);
    hb.pw1 = cv.take<float>((size_t)hb.slabs * nc * Cp);
    hb.pb1 = cv.take<float>((size_t)hb.slabs * nc);
  }
  return align_up(cv.off, 256);
}

// Minibatch negatives (pnce_head_mb_fwd) only: the gather's partial sums of squares of the raw patches, which mark a
// non-finite patch for k_head_mb_guard.  Carved AFTER carve_head's layout, so that pnce_head_bwd_ex's carve sees the
// offsets the forward used; with base == nullptr only the size is computed.
static size_t carve_head_mb(const pnce_layer_t* layers, int n_layers, int B, void* base, Params* pg) {
  Carver cv(base);
  for (int l = 0; l < n_layers; ++l) {
    const size_t Ppad = (layers[l].P + 127) / 128 * 128, nchunk = (layers[l].C + 31) / 32;
    float* qss = cv.take<float>((size_t)B * nchunk * Ppad);
    float* kss = cv.take<float>((size_t)B * nchunk * Ppad);
    if (pg != nullptr) { pg->L[l].qss = qss; pg->L[l].kss = kss; }
  }
  return align_up(cv.off, 256);
}

static int launch_gemm(GemmLaunch& g, cudaStream_t st) {
  g.dbg = g_dbg.gemm_dbg;
  long long acc = 0;
  for (int i = 0; i < g.n; ++i) { g.start[i] = acc; acc += g.pr[i].tiles; }
  g.start[g.n] = acc;
  if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
  if (!g_dbg.no_persist) {
    // persistent: one CTA per SM, double-buffered TMEM accumulator (tile n+1's MMAs under tile n's epilogue)
    int nsm = 0;
    int rc = sm_count(&nsm);
    if (rc != PNCE_OK) return rc;
    long long grid = g_dbg.persist_ctas > 0 ? g_dbg.persist_ctas : nsm;
    if (grid > acc) grid = acc;
    rc = set_smem(k_gemm_tc_p, kGpSmemBytes);
    if (rc != PNCE_OK) return rc;
    launch_k(k_gemm_tc_p, (unsigned)grid, kGpThreads, kGpSmemBytes, st, g);
    PNCE_CUDA(cudaGetLastError());
    return PNCE_OK;
  }
  int rc = set_smem(k_gemm_tc, kGemmSmemBytes);
  if (rc != PNCE_OK) return rc;
  launch_k(k_gemm_tc, (unsigned)acc, kTcThreads, kGemmSmemBytes, st, g);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int check_head_args(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch,
                           int dtype, int nc, int math_mode, void* ws, bool bwd) {
  int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (heads == nullptr || dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (math_mode != PNCE_MATH_TC_BF16X3 && math_mode != PNCE_MATH_TC_BF16) return PNCE_ERR_UNSUPPORTED;
  if (!head_shapes_ok(layers, n_layers, nc)) return PNCE_ERR_UNSUPPORTED;
  for (int l = 0; l < n_layers; ++l) {
    const pnce_head_t& h = heads[l];
    if (!h.w1 || !h.b1 || !h.w2 || !h.b2) return PNCE_ERR_ARG;
    if (bwd && (!h.dw1 || !h.db1 || !h.dw2 || !h.db2)) return PNCE_ERR_ARG;
  }
  rc = check_alignment(layers, n_layers, dtype, bwd);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  return PNCE_OK;
}

}  // namespace pnce

int pnce_head_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, int nc, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!head_shapes_ok(layers, n_layers, nc)) return PNCE_ERR_UNSUPPORTED;
  *bytes = carve_head(layers, n_layers, batch, nc, true, nullptr, nullptr);
  return PNCE_OK;
}

// The Params fields of a head forward that the carve leaves open (both parts below read them).
static void head_fwd_setup(HeadPlan& hp, int batch, int dtype, int layout, int math_mode, float temperature,
                           float* loss_out, int* nonfinite, bool mb) {
  Params& pg = hp.pg;
  Params& pl = hp.pl;
  pg.dtype = pl.dtype = dtype;
  pg.math = pl.math = math_mode;
  pg.tau = pl.tau = temperature;
  pl.loss_out = loss_out;
  pg.nonfinite = pl.nonfinite = nonfinite;
  pg.b0 = pl.b0 = 0; pg.bn = pl.bn = batch;
  pg.nhwc = layout == PNCE_LAYOUT_NHWC ? 1 : 0;               // the maps; the head's output (pl) has no layout
  pl.mb = mb ? 1 : 0;
  pl.trace = g_dbg.trace;
}

// Keys part of the head forward: steps 1-4b, up to the head's output on both sides.  The key side of the second GEMM
// (khi / klo, k2hi / k2lo, kss) and k_head_mb_guard's key marks go to the blobs of kdst's layers: the virtual layers'
// own (hp.pl), or a slot of the global-negatives workspace (pnce_head_mb_shard_keys).
static int head_fwd_keys(HeadPlan& hp, const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch,
                         int nc, bool x3, bool mb, int* nonfinite, const Params& kdst, cudaStream_t st) {
  Params& pg = hp.pg;
  Params& pl = hp.pl;
  int rc = PNCE_OK;
  // 1. ids -> sorted slots; weights -> operand blobs
  const bool fold = gather_tc_folds(pg);                      // small problems: the gather CTAs sort the ids themselves
  if (!fold) rc = launch_prep(pg, st);
  if (rc != PNCE_OK) return rc;
  {
    static thread_local WprepLaunch wl;
    memset(&wl, 0, sizeof(wl));
    int blocks = 0;
    auto add = [&](const float* w, __nv_bfloat16* hi, __nv_bfloat16* lo, int R, int Cw, int N, int K, int tr) {
      WprepJob& j = wl.job[wl.n];
      j.w = w; j.hi = hi; j.lo = lo; j.R = R; j.Cw = Cw; j.N = N; j.K = K; j.transpose = tr;
      wl.start[wl.n++] = blocks;
      blocks += (N / 8) * (K / 8);
    };
    for (int l = 0; l < n_layers; ++l) {
      const HeadLayerBufs& hb = hp.hb[l];
      const int C = layers[l].C, Cp = pg.L[l].Cp;
      add(heads[l].w1, hb.w1[0], hb.w1[1], nc, C, nc, Cp, 0);     // B[n][k] = W1[n][k]      (H = X W1^T)
      add(heads[l].w1, hb.w1t[0], hb.w1t[1], nc, C, Cp, nc, 1);   // B[c][j] = W1[j][c]      (dX = dH W1)
      add(heads[l].w2, hb.w2[0], hb.w2[1], nc, nc, nc, nc, 0);    // B[n][k] = W2[n][k]      (Y = H W2^T)
      add(heads[l].w2, hb.w2t[0], hb.w2t[1], nc, nc, nc, nc, 1);  // B[j][i] = W2[i][j]      (dH = dY W2)
    }
    wl.start[wl.n] = blocks;
    launch_k(k_wprep, (unsigned)blocks, 64, 0, st, wl);
    PNCE_CUDA(cudaGetLastError());
  }
  // 2. raw patches of both sides as row blobs
  rc = launch_gather_tc(pg, st, fold);
  if (rc != PNCE_OK) return rc;
  // 3. H = relu(X W1^T + b1), both sides
  static thread_local GemmLaunch g;
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  g.err = nonfinite ? nonfinite + 1 : nullptr;
  for (int l = 0; l < n_layers; ++l) {
    const HeadLayerBufs& hb = hp.hb[l];
    const LayerDev& G = pg.L[l];
    for (int side = 0; side < 2; ++side) {
      GemmProb& pr = g.pr[g.n++];
      pr.a_hi = side ? hb.xq[0] : hb.xk[0]; pr.a_lo = side ? hb.xq[1] : hb.xk[1];
      pr.b_hi = hb.w1[0]; pr.b_lo = hb.w1[1];
      pr.bias = heads[l].b1;
      pr.K = G.Cp; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_H;
      pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = G.C;
      pr.o_hi = side ? hb.hq[0] : hb.hk[0]; pr.o_lo = side ? hb.hq[1] : hb.hk[1];
    }
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  // 4. Y = H W2^T + b2 straight into the operand formats of k_loss_tc
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  g.err = nonfinite ? nonfinite + 1 : nullptr;
  for (int l = 0; l < n_layers; ++l) {
    const HeadLayerBufs& hb = hp.hb[l];
    const LayerDev& G = pg.L[l];
    const LayerDev& V = pl.L[l];
    const LayerDev& K = kdst.L[l];
    for (int side = 0; side < 2; ++side) {
      GemmProb& pr = g.pr[g.n++];
      pr.a_hi = side ? hb.hq[0] : hb.hk[0]; pr.a_lo = side ? hb.hq[1] : hb.hk[1];
      pr.b_hi = hb.w2[0]; pr.b_lo = hb.w2[1];
      pr.bias = heads[l].b2;
      pr.K = nc; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = side ? GM_YQ : GM_YK;
      pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = nc;
      if (side) { pr.o_hi = V.qhi; pr.o_lo = V.qlo; pr.ss = V.qss; }
      else { pr.k_hi = K.khi; pr.k_lo = K.klo; pr.k2_hi = K.k2hi; pr.k2_lo = K.k2lo; pr.ss = K.kss; }
    }
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  if (mb) {
    // 4b. a non-finite raw patch -> a non-finite row / key of the head's output (the layer's group guard)
    static thread_local HeadGuardLaunch gl;
    memset(&gl, 0, sizeof(gl));
    gl.B = batch;
    long long most = 0;
    for (int l = 0; l < n_layers; ++l) {
      const LayerDev& G = pg.L[l];
      const LayerDev& V = pl.L[l];
      HeadGuardLayer& h = gl.L[l];
      h.xqss = G.qss; h.xkss = G.kss; h.yqss = V.qss; h.ykss = kdst.L[l].kss;
      h.xq_hi = hp.hb[l].xq[0]; h.xq_lo = x3 ? hp.hb[l].xq[1] : nullptr;
      h.P = G.P; h.Ppad = G.Ppad; h.Cp8 = G.Cp / 8; h.nchunk = G.nchunk; h.ncy = nc / 32;
      if ((long long)batch * G.Ppad > most) most = (long long)batch * G.Ppad;
    }
    launch_k(k_head_mb_guard, dim3((unsigned)((most + kThreads - 1) / kThreads), (unsigned)n_layers), kThreads, 0, st, gl);
    PNCE_CUDA(cudaGetLastError());
  }
  return PNCE_OK;
}

// Loss part of the head forward: step 5, logits / diagonal CE / d loss / d Y (as a row blob) on the head's output.
static int head_fwd_loss(Params& pl, int batch, cudaStream_t st) {
  int ctas = 0;
  for (int l = 0; l < pl.n_layers; ++l) ctas += pl.L[l].Ppad / 128;
  pl.total_ctas = (unsigned)(batch * ctas);
  return launch_loss_tc(pl, st);
}

// mb: minibatch negatives -- the loss launch is k_loss_tc_mb on the same virtual layers (see pnce_head_mb_fwd)
static int head_fwd_impl(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                         int layout, int nc, float temperature, int math_mode, void* ws, size_t ws_bytes, float* loss_out,
                         int* nonfinite, void* stream, bool mb = false) {
  int rc = check_head_args(layers, heads, n_layers, batch, dtype, nc, math_mode, ws, false);
  if (rc != PNCE_OK) return rc;
  if (loss_out == nullptr || !(temperature > 0.f)) return PNCE_ERR_ARG;
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  static thread_local HeadPlan hp;
  size_t need = carve_head(layers, n_layers, batch, nc, x3, ws, &hp);
  if (mb) need += carve_head_mb(layers, n_layers, batch, static_cast<unsigned char*>(ws) + need, &hp.pg);
  if (need > ws_bytes) return PNCE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  head_fwd_setup(hp, batch, dtype, layout, math_mode, temperature, loss_out, nonfinite, mb);
  rc = head_fwd_keys(hp, layers, heads, n_layers, batch, nc, x3, mb, nonfinite, hp.pl, st);
  if (rc != PNCE_OK) return rc;
  return head_fwd_loss(hp.pl, batch, st);
}

// phases: bit 0 = head backward proper (dH, dX, weight / bias gradients), bit 1 = dense d tgt_feat
static int head_bwd_phases(int phases, const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch,
                           int dtype, int nc, int math_mode, void* ws, size_t ws_bytes, const float* grad_out,
                           void* stream, int layout = PNCE_LAYOUT_NCHW) {
  int rc = check_head_args(layers, heads, n_layers, batch, dtype, nc, math_mode, ws, (phases & 2) != 0);
  if (rc != PNCE_OK) return rc;
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (phases < 1 || phases > 3) return PNCE_ERR_ARG;
  if (phases & 1)
    for (int l = 0; l < n_layers; ++l)
      if (!heads[l].dw1 || !heads[l].db1 || !heads[l].dw2 || !heads[l].db2) return PNCE_ERR_ARG;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  static thread_local HeadPlan hp;
  if (carve_head(layers, n_layers, batch, nc, x3, ws, &hp) > ws_bytes) return PNCE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Params& pg = hp.pg;
  pg.dtype = dtype;
  pg.grad_out = grad_out;
  pg.nhwc = layout == PNCE_LAYOUT_NHWC ? 1 : 0;
  if (!(phases & 1)) return launch_dense(pg, st);
  static thread_local GemmLaunch g;
  // 1. dH = (dY W2) * [H > 0]
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  for (int l = 0; l < n_layers; ++l) {
    const HeadLayerBufs& hb = hp.hb[l];
    const LayerDev& G = pg.L[l];
    const LayerDev& V = hp.pl.L[l];
    GemmProb& pr = g.pr[g.n++];
    pr.a_hi = V.dyhi; pr.a_lo = V.dylo; pr.b_hi = hb.w2t[0]; pr.b_lo = hb.w2t[1];
    pr.K = nc; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_DH;
    pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = nc;
    pr.o_hi = hb.dh[0]; pr.o_lo = hb.dh[1]; pr.mask_hi = hb.hq[0];
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  // 2. dX = dH W1 -> the transposed fp32 rows the dense backward reads
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  for (int l = 0; l < n_layers; ++l) {
    const HeadLayerBufs& hb = hp.hb[l];
    const LayerDev& G = pg.L[l];
    GemmProb& pr = g.pr[g.n++];
    pr.a_hi = hb.dh[0]; pr.a_lo = hb.dh[1]; pr.b_hi = hb.w1t[0]; pr.b_lo = hb.w1t[1];
    pr.K = nc; pr.N = G.Cp; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_DX;
    pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = G.C;
    pr.outT = G.dxT; pr.rm = pg.nhwc;
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  // 3. weight / bias gradients: split-K partials, then a deterministic reduce scaled by the upstream
  static thread_local WgradLaunch wg;
  memset(&wg, 0, sizeof(wg));
  wg.x3 = x3 ? 1 : 0;
  long long acc = 0;
  for (int l = 0; l < n_layers; ++l) {
    const HeadLayerBufs& hb = hp.hb[l];
    const LayerDev& G = pg.L[l];
    const LayerDev& V = hp.pl.L[l];
    const int tiles = batch * (G.Ppad / 128);
    for (int which = 0; which < 2; ++which) {
      WgradProb& pr = wg.pr[wg.n];
      pr.a_hi = which ? hb.dh[0] : V.dyhi; pr.a_lo = which ? hb.dh[1] : V.dylo;
      pr.b_hi = which ? hb.xq[0] : hb.hq[0]; pr.b_lo = which ? hb.xq[1] : hb.hq[1];
      pr.NA = nc; pr.N = which ? G.Cp : nc; pr.tiles = tiles; pr.slabs = hb.slabs;
      pr.partial = which ? hb.pw1 : hb.pw2; pr.pbias = which ? hb.pb1 : hb.pb2;
      wg.start[wg.n++] = acc;
      acc += (long long)hb.slabs * (nc / 128);
    }
  }
  wg.start[wg.n] = acc;
  rc = set_smem(k_wgrad_tc, kWgSmemBytes);
  if (rc != PNCE_OK) return rc;
  launch_k(k_wgrad_tc, (unsigned)acc, kTcThreads, kWgSmemBytes, st, wg);
  PNCE_CUDA(cudaGetLastError());
  {
    static thread_local WreduceLaunch rl;
    memset(&rl, 0, sizeof(rl));
    rl.grad_out = grad_out;
    int blocks = 0;
    for (int l = 0; l < n_layers; ++l) {
      const HeadLayerBufs& hb = hp.hb[l];
      const LayerDev& G = pg.L[l];
      for (int which = 0; which < 2; ++which) {
        WreduceJob& j = rl.job[rl.n];
        j.partial = which ? hb.pw1 : hb.pw2; j.pbias = which ? hb.pb1 : hb.pb2;
        j.dw = which ? heads[l].dw1 : heads[l].dw2; j.db = which ? heads[l].db1 : heads[l].db2;
        j.NA = nc; j.N = which ? G.Cp : nc; j.Nout = which ? G.C : nc; j.slabs = hb.slabs;
        rl.start[rl.n++] = blocks;
        blocks += (int)(((long long)nc * j.N + nc + kThreads - 1) / kThreads);
      }
    }
    rl.start[rl.n] = blocks;
    launch_k(k_wreduce, (unsigned)blocks, kThreads, 0, st, rl);
    PNCE_CUDA(cudaGetLastError());
  }
  // 4. dense d tgt_feat (zero fill + sampled positions), scaled by the upstream gradient
  if (!(phases & 2)) return PNCE_OK;
  return launch_dense(pg, st);
}

int pnce_head_fwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                  int nc, float temperature, int math_mode, void* ws, size_t ws_bytes, float* loss_out,
                  int* nonfinite, void* stream) {
  return head_fwd_impl(layers, heads, n_layers, batch, dtype, PNCE_LAYOUT_NCHW, nc, temperature, math_mode, ws, ws_bytes,
                       loss_out, nonfinite, stream);
}
int pnce_head_fwd_ex(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int nc, float temperature, int math_mode, void* ws, size_t ws_bytes, float* loss_out,
                     int* nonfinite, void* stream) {
  return head_fwd_impl(layers, heads, n_layers, batch, dtype, layout, nc, temperature, math_mode, ws, ws_bytes, loss_out,
                       nonfinite, stream);
}
int pnce_head_bwd_ex(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int phases, int nc, int math_mode, void* ws, size_t ws_bytes, const float* grad_out, void* stream) {
  return head_bwd_phases(phases, layers, heads, n_layers, batch, dtype, nc, math_mode, ws, ws_bytes, grad_out, stream, layout);
}
int pnce_head_bwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                  int nc, int math_mode, void* ws, size_t ws_bytes, const float* grad_out, void* stream) {
  return head_bwd_phases(3, layers, heads, n_layers, batch, dtype, nc, math_mode, ws, ws_bytes, grad_out, stream);
}
int pnce_head_bwd_params(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                         int nc, int math_mode, void* ws, size_t ws_bytes, const float* grad_out, void* stream) {
  return head_bwd_phases(1, layers, heads, n_layers, batch, dtype, nc, math_mode, ws, ws_bytes, grad_out, stream);
}
int pnce_head_bwd_dense(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                        int nc, int math_mode, void* ws, size_t ws_bytes, const float* grad_out, void* stream) {
  return head_bwd_phases(2, layers, heads, n_layers, batch, dtype, nc, math_mode, ws, ws_bytes, grad_out, stream);
}

// ---- netF head with minibatch negatives ----------------------------------------------------------------------------
// The head's second GEMM writes the key side (khi / klo, k2hi / k2lo, kss) per image in the key-blocked layout of the
// gather, so the batch's key blobs are the one blob of B * Ppad keys k_loss_tc_mb walks.  k_loss_tc_mb reads nothing
// carve_head lacks on the virtual layers: qss / kss ([B][nc / 32][Ppad], key norms folded per key block), qinv (B * P),
// partial (B * max(Ppad / 128, 2) >= B * nparts), lossimg / valid (n_layers * B) and the counter; it writes d loss / d Y
// into dyhi / dylo (dxT == nullptr: the epilogue's head branch stores no fp32 rows), and its last CTA zeroes the dY rows
// of a guarded layer (valid = 0 for every image).  kinv is not used in this mode.  The one addition is carve_head_mb's
// raw-patch sums of squares for k_head_mb_guard, after carve_head's layout: pnce_head_bwd_ex reads the workspace
// unchanged.
static bool head_mb_shapes_ok(const pnce_layer_t* layers, int n_layers, int B, int nc) {
  if (!head_shapes_ok(layers, n_layers, nc)) return false;
  for (int l = 0; l < n_layers; ++l)
    if (!mb_keys_ok(B, layers[l].P)) return false;
  return true;
}

int pnce_head_mb_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, int nc, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!head_mb_shapes_ok(layers, n_layers, batch, nc)) return PNCE_ERR_UNSUPPORTED;
  *bytes = carve_head(layers, n_layers, batch, nc, true, nullptr, nullptr) + carve_head_mb(layers, n_layers, batch, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_head_mb_fwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int nc, float temperature, int math_mode, void* ws, size_t ws_bytes, float* loss_out,
                     int* nonfinite, void* stream) {
  if (math_mode == PNCE_MATH_SIMT_F32) return PNCE_ERR_UNSUPPORTED;
  const int rc = check_layers(layers, n_layers, batch);
  if (rc != PNCE_OK) return rc;
  if (!head_mb_shapes_ok(layers, n_layers, batch, nc)) return PNCE_ERR_UNSUPPORTED;
  return head_fwd_impl(layers, heads, n_layers, batch, dtype, layout, nc, temperature, math_mode, ws, ws_bytes, loss_out,
                       nonfinite, stream, true);
}

// ---- netF head with global negatives: minibatch negatives over the shards of every rank ------------------------------
// Workspace: the prefix pnce_head_mb_workspace_bytes(batch_local) -- carve_head, then carve_head_mb, exactly what
// pnce_head_mb_fwd lays out and pnce_head_bwd_ex reads -- followed by `world` slots in the format of pnce_mb_shard_*
// (carve_mb_slot on the virtual layers, C = nc).  The second GEMM writes this rank's keys straight into its slot and
// k_loss_tc_mb_gn reads every slot's; carve_head's own key blobs of the virtual layers stay unused in this mode (trimming
// them would move the offsets the backward reads).
//
// The query flags: k_mb_qbad on the virtual layers, i.e. "a NaN among the partial sums of squares of a query row of the
// head's output".  That is exactly the loss kernel's own row test (badq: the sum of the row's partials is NaN), because
// every partial is finite or NaN: libpnce.so runs k_gemm_tc_p (g_dbg.no_persist is a constexpr 0), whose GM_YQ / GM_YK
// epilogue stores NaN for a 32-channel chunk whose sum of squares is not finite (gemm_tc_persist.cuh, isfinite(ssum));
// k_head_mb_guard stores NaN on chunk 0 for a non-finite raw patch; padding rows are exactly 0.  (k_gemm_tc, reachable
// only through the experiment build's knob 6, stores +Inf for an overflowing chunk: not covered.)  An unflagged row and
// key then have norms below 5.2e19, and their logit is non-finite only when q . k overflows fp32, i.e. both norms above
// 6.5e18: the one window where the owning rank guards alone (DESIGN.md 4.14).

// The envelope of the GLOBAL batch and the slot geometry: *prefix, the slots' offset; *slot_bytes, their stride; vl, the
// virtual layers (C = nc) the slots are carved on.  No CUDA call.
static int head_shard_geometry(const pnce_layer_t* layers, int n_layers, int batch_local, int world, int nc,
                               pnce_layer_t* vl, size_t* prefix, size_t* slot_bytes) {
  const int rc = global_batch_check(world, batch_local, [&](int B) {
    return head_mb_shapes_ok(layers, n_layers, B, nc) ? PNCE_OK : PNCE_ERR_UNSUPPORTED;
  });
  if (rc != PNCE_OK) return rc;
  for (int l = 0; l < n_layers; ++l) {
    vl[l] = layers[l];
    vl[l].C = nc;
  }
  *prefix = carve_head(layers, n_layers, batch_local, nc, true, nullptr, nullptr) +
            carve_head_mb(layers, n_layers, batch_local, nullptr, nullptr);
  *slot_bytes = carve_mb_slot(vl, n_layers, batch_local, true, nullptr, nullptr);
  return PNCE_OK;
}

// The checks of the two shard calls, all before any CUDA call, then the carve of the prefix into hp.  *prefix,
// *slot_bytes, vl: head_shard_geometry's.
static int head_shard_plan(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch_local,
                           int dtype, int layout, int nc, int world, int rank, int math_mode, void* ws, size_t ws_bytes,
                           HeadPlan& hp, pnce_layer_t* vl, size_t* prefix, size_t* slot_bytes) {
  int rc = check_layers(layers, n_layers, batch_local);
  if (rc != PNCE_OK) return rc;
  if (world < 1 || rank < 0 || rank >= world) return PNCE_ERR_ARG;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (math_mode < PNCE_MATH_SIMT_F32 || math_mode > PNCE_MATH_TC_BF16) return PNCE_ERR_ARG;
  if (heads == nullptr) return PNCE_ERR_ARG;
  for (int l = 0; l < n_layers; ++l)
    if (!heads[l].w1 || !heads[l].b1 || !heads[l].w2 || !heads[l].b2) return PNCE_ERR_ARG;
  if (math_mode == PNCE_MATH_SIMT_F32) return PNCE_ERR_UNSUPPORTED;
  rc = head_shard_geometry(layers, n_layers, batch_local, world, nc, vl, prefix, slot_bytes);
  if (rc != PNCE_OK) return rc;
  rc = check_alignment(layers, n_layers, dtype, false);
  if (rc != PNCE_OK) return rc;
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  if (*prefix + (size_t)world * *slot_bytes > ws_bytes) return PNCE_ERR_WORKSPACE;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  const size_t used = carve_head(layers, n_layers, batch_local, nc, x3, ws, &hp);
  carve_head_mb(layers, n_layers, batch_local, static_cast<unsigned char*>(ws) + used, &hp.pg);
  return PNCE_OK;
}

int pnce_head_mb_shard_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch_local, int world, int nc,
                                       size_t* bytes, size_t* slot_offset, size_t* slot_bytes) {
  if (bytes == nullptr || slot_offset == nullptr || slot_bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_layers(layers, n_layers, batch_local);
  if (rc != PNCE_OK) return rc;
  if (world < 1) return PNCE_ERR_ARG;
  pnce_layer_t vl[PNCE_MAX_LAYERS];
  rc = head_shard_geometry(layers, n_layers, batch_local, world, nc, vl, slot_offset, slot_bytes);
  if (rc != PNCE_OK) return rc;
  *bytes = *slot_offset + (size_t)world * *slot_bytes;
  return PNCE_OK;
}

int pnce_head_mb_shard_keys(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch_local,
                            int dtype, int layout, int nc, int world, int rank, int math_mode, void* ws,
                            size_t ws_bytes, int* nonfinite, void* stream) {
  static thread_local HeadPlan hp;
  static thread_local Params kd;                               // slot `rank`: where the keys and the flags go
  pnce_layer_t vl[PNCE_MAX_LAYERS];
  size_t prefix = 0, slot_bytes = 0;
  int rc = head_shard_plan(layers, heads, n_layers, batch_local, dtype, layout, nc, world, rank, math_mode, ws, ws_bytes,
                           hp, vl, &prefix, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  memset(&kd, 0, sizeof(kd));
  carve_mb_slot(vl, n_layers, batch_local, x3, static_cast<unsigned char*>(ws) + prefix + (size_t)rank * slot_bytes, &kd);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  head_fwd_setup(hp, batch_local, dtype, layout, math_mode, 1.0f, nullptr, nonfinite, true);
  rc = head_fwd_keys(hp, layers, heads, n_layers, batch_local, nc, x3, true, nonfinite, kd, st);
  if (rc != PNCE_OK) return rc;
  // this rank's "a query row is non-finite" flags, next to its keys (see above for why k_mb_qbad is exact here)
  return launch_mb_qbad(hp.pl, const_cast<int*>(kd.qbad), st);
}

int pnce_head_mb_shard_loss(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch_local,
                            int dtype, int layout, int nc, int world, int rank, float temperature, int math_mode,
                            void* ws, size_t ws_bytes, float* loss_out, int* nonfinite, void* stream) {
  static thread_local HeadPlan hp;
  pnce_layer_t vl[PNCE_MAX_LAYERS];
  size_t prefix = 0, slot_bytes = 0;
  int rc = head_shard_plan(layers, heads, n_layers, batch_local, dtype, layout, nc, world, rank, math_mode, ws, ws_bytes,
                           hp, vl, &prefix, &slot_bytes);
  if (rc != PNCE_OK) return rc;
  if (loss_out == nullptr || !(temperature > 0.f)) return PNCE_ERR_ARG;
  head_fwd_setup(hp, batch_local, dtype, layout, math_mode, temperature, loss_out, nonfinite, true);
  // the virtual layers' key blobs and qbad: slot 0 of `world` (point_at_slots)
  carve_mb_slot(vl, n_layers, batch_local, math_mode == PNCE_MATH_TC_BF16X3, static_cast<unsigned char*>(ws) + prefix,
                &hp.pl);
  point_at_slots(hp.pl, world, rank, slot_bytes);
  return head_fwd_loss(hp.pl, batch_local, static_cast<cudaStream_t>(stream));
}


// ---- PatchSampleF(use_mlp=True) as a module of its own ------------------------------------------------------------
namespace pnce {

struct NetfPlan {
  Params pg;                                   // the maps: gather of raw patches, dense backward of dX
  HeadLayerBufs hb[PNCE_MAX_LAYERS];           // xq = X blob, hq = H blob, dh = dH blob, weight blobs, split-K partials
  __nv_bfloat16* dy[PNCE_MAX_LAYERS][2];       // d loss / d Y blob (hi, lo)
};

static size_t carve_netf(const pnce_sample_t* sm, int n, int B, int nc, bool x3, void* ws, NetfPlan* out) {
  Carver cv(ws);
  NetfPlan local;
  NetfPlan* np = out ? out : &local;
  memset(np, 0, sizeof(NetfPlan));
  Params& pg = np->pg;
  pg.n_layers = n;
  pg.B = B;
  pg.side0 = 1;                                // one side only: the maps play the "tgt" role of the fused kernels
  const int nparts = x3 ? 2 : 1;
  for (int l = 0; l < n; ++l) {
    const pnce_sample_t& a = sm[l];
    LayerDev& G = pg.L[l];
    HeadLayerBufs& hb = np->hb[l];
    const int Ppad = (a.P + 127) / 128 * 128, Cp = (a.C + 31) / 32 * 32;
    G.tgt = a.feat; G.dtgt = a.dfeat;
    G.ids = reinterpret_cast<const long long*>(a.ids);
    G.C = a.C; G.HW = a.H * a.W; G.P = a.P;
    G.ntiles = (a.P + kRowTile - 1) / kRowTile;
    G.sorted = 1;
    G.Cp = Cp; G.Ppad = Ppad; G.nchunk = Cp / 32; G.nparts = Ppad / 128;
    G.head_src_rows = 1;
    G.sid = cv.take<int>(a.P);
    G.perm = cv.take<int>(a.P);
    G.rank = cv.take<int>(a.P);
    G.cslot = cv.take<int>((size_t)(G.HW + kTilePos - 1) / kTilePos + 1);
    G.dxpitch = Ppad;
    G.dxT = cv.take<float>((size_t)B * a.C * Ppad);
    const size_t xblob = (size_t)B * Ppad * Cp, yblob = (size_t)B * Ppad * nc;
    for (int k = 0; k < nparts; ++k) {
      hb.xq[k] = cv.take<__nv_bfloat16>(xblob);
      hb.hq[k] = cv.take<__nv_bfloat16>(yblob);
      hb.dh[k] = cv.take<__nv_bfloat16>(yblob);
      np->dy[l][k] = cv.take<__nv_bfloat16>(yblob);
      hb.w1[k] = cv.take<__nv_bfloat16>((size_t)nc * Cp);
      hb.w1t[k] = cv.take<__nv_bfloat16>((size_t)nc * Cp);
      hb.w2[k] = cv.take<__nv_bfloat16>((size_t)nc * nc);
      hb.w2t[k] = cv.take<__nv_bfloat16>((size_t)nc * nc);
    }
    G.qhi = hb.xq[0]; G.qlo = hb.xq[1];
    const int tiles = B * (Ppad / 128);
    hb.slabs = tiles < 8 ? tiles : 8;
    hb.pw2 = cv.take<float>((size_t)hb.slabs * nc * nc);
    hb.pb2 = cv.take<float>((size_t)hb.slabs * nc);
    hb.pw1 = cv.take<float>((size_t)hb.slabs * nc * Cp);
    hb.pb1 = cv.take<float>((size_t)hb.slabs * nc);
  }
  return align_up(cv.off, 256);
}

static int check_netf(const pnce_sample_t* sm, const pnce_head_t* heads, int n, int batch, int dtype, int layout, int nc,
                      int math_mode, void* ws) {
  int rc = check_samples(sm, n, batch, dtype);
  if (rc != PNCE_OK) return rc;
  if (heads == nullptr) return PNCE_ERR_ARG;
  if (layout != PNCE_LAYOUT_NCHW && layout != PNCE_LAYOUT_NHWC) return PNCE_ERR_ARG;
  if (math_mode != PNCE_MATH_TC_BF16X3 && math_mode != PNCE_MATH_TC_BF16) return PNCE_ERR_UNSUPPORTED;
  if (nc != 128 && nc != 256) return PNCE_ERR_UNSUPPORTED;
  for (int l = 0; l < n; ++l) {
    if (sm[l].P > 1024 || sm[l].C > 256) return PNCE_ERR_UNSUPPORTED;
    const pnce_head_t& h = heads[l];
    if (!h.w1 || !h.b1 || !h.w2 || !h.b2) return PNCE_ERR_ARG;
  }
  if (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 255u)) return PNCE_ERR_WORKSPACE;
  return PNCE_OK;
}

}  // namespace pnce

int pnce_netf_workspace_bytes(const pnce_sample_t* maps, int n_maps, int batch, int nc, size_t* bytes) {
  if (bytes == nullptr) return PNCE_ERR_ARG;
  int rc = check_samples(maps, n_maps, batch, PNCE_F32);
  if (rc != PNCE_OK) return rc;
  if (nc != 128 && nc != 256) return PNCE_ERR_UNSUPPORTED;
  for (int l = 0; l < n_maps; ++l)
    if (maps[l].P > 1024 || maps[l].C > 256) return PNCE_ERR_UNSUPPORTED;
  *bytes = carve_netf(maps, n_maps, batch, nc, true, nullptr, nullptr);
  return PNCE_OK;
}

int pnce_netf_fwd(const pnce_sample_t* maps, const pnce_head_t* heads, int n_maps, int batch, int dtype, int layout,
                  int nc, int math_mode, void* ws, size_t ws_bytes, int* dev_status, void* stream) {
  int rc = check_netf(maps, heads, n_maps, batch, dtype, layout, nc, math_mode, ws);
  if (rc != PNCE_OK) return rc;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  static thread_local NetfPlan np;
  if (carve_netf(maps, n_maps, batch, nc, x3, ws, &np) > ws_bytes) return PNCE_ERR_WORKSPACE;
  Params& pg = np.pg;
  for (int l = 0; l < n_maps; ++l) {
    if (maps[l].feat == nullptr || maps[l].rows == nullptr || maps[l].inv == nullptr) return PNCE_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(maps[l].feat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
    if (reinterpret_cast<uintptr_t>(maps[l].rows) & 15u) return PNCE_ERR_ALIGN;
  }
  pg.dtype = dtype;
  pg.math = math_mode;
  pg.nhwc = layout == PNCE_LAYOUT_NHWC ? 1 : 0;
  pg.b0 = 0; pg.bn = batch;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // 1. ids -> sorted slots; weights -> operand blobs (plain and transposed: the backward needs both)
  const bool fold = gather_tc_folds(pg);                      // small problems: the gather CTAs sort the ids themselves
  if (!fold) rc = launch_prep(pg, st);
  if (rc != PNCE_OK) return rc;
  {
    static thread_local WprepLaunch wl;
    memset(&wl, 0, sizeof(wl));
    int blocks = 0;
    auto add = [&](const float* w, __nv_bfloat16* hi, __nv_bfloat16* lo, int R, int Cw, int N, int K, int tr) {
      WprepJob& j = wl.job[wl.n];
      j.w = w; j.hi = hi; j.lo = lo; j.R = R; j.Cw = Cw; j.N = N; j.K = K; j.transpose = tr;
      wl.start[wl.n++] = blocks;
      blocks += (N / 8) * (K / 8);
    };
    for (int l = 0; l < n_maps; ++l) {
      const HeadLayerBufs& hb = np.hb[l];
      const int C = maps[l].C, Cp = pg.L[l].Cp;
      add(heads[l].w1, hb.w1[0], hb.w1[1], nc, C, nc, Cp, 0);
      add(heads[l].w1, hb.w1t[0], hb.w1t[1], nc, C, Cp, nc, 1);
      add(heads[l].w2, hb.w2[0], hb.w2[1], nc, nc, nc, nc, 0);
      add(heads[l].w2, hb.w2t[0], hb.w2t[1], nc, nc, nc, nc, 1);
    }
    wl.start[wl.n] = blocks;
    launch_k(k_wprep, (unsigned)blocks, 64, 0, st, wl);
    PNCE_CUDA(cudaGetLastError());
  }
  // 2. raw patches as the X row blob (sorted-slot order)
  rc = launch_gather_tc(pg, st, fold);
  if (rc != PNCE_OK) return rc;
  // 3. H = relu(X W1^T + b1)
  static thread_local GemmLaunch g;
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  g.err = dev_status;
  for (int l = 0; l < n_maps; ++l) {
    const HeadLayerBufs& hb = np.hb[l];
    const LayerDev& G = pg.L[l];
    GemmProb& pr = g.pr[g.n++];
    pr.a_hi = hb.xq[0]; pr.a_lo = hb.xq[1]; pr.b_hi = hb.w1[0]; pr.b_lo = hb.w1[1];
    pr.bias = heads[l].b1;
    pr.K = G.Cp; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_H;
    pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = G.C;
    pr.o_hi = hb.hq[0]; pr.o_lo = hb.hq[1];
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  // 4. Y = H W2^T + b2, L2-normalised, as fp32 rows in the caller's row order
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  g.err = dev_status;
  for (int l = 0; l < n_maps; ++l) {
    const HeadLayerBufs& hb = np.hb[l];
    const LayerDev& G = pg.L[l];
    GemmProb& pr = g.pr[g.n++];
    pr.a_hi = hb.hq[0]; pr.a_lo = hb.hq[1]; pr.b_hi = hb.w2[0]; pr.b_lo = hb.w2[1];
    pr.bias = heads[l].b2;
    pr.K = nc; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_YROWS;
    pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = nc;
    pr.rows_out = maps[l].rows; pr.inv_out = maps[l].inv; pr.perm = G.perm;
  }
  return launch_gemm(g, st);
}

int pnce_netf_bwd(const pnce_sample_t* maps, const pnce_head_t* heads, int n_maps, int batch, int dtype, int layout,
                  int nc, int math_mode, void* ws, size_t ws_bytes, int* dev_status, void* stream) {
  int rc = check_netf(maps, heads, n_maps, batch, dtype, layout, nc, math_mode, ws);
  if (rc != PNCE_OK) return rc;
  const bool x3 = math_mode == PNCE_MATH_TC_BF16X3;
  static thread_local NetfPlan np;
  if (carve_netf(maps, n_maps, batch, nc, x3, ws, &np) > ws_bytes) return PNCE_ERR_WORKSPACE;
  Params& pg = np.pg;
  bool dense = true;
  for (int l = 0; l < n_maps; ++l) {
    const pnce_head_t& h = heads[l];
    if (!h.dw1 || !h.db1 || !h.dw2 || !h.db2) return PNCE_ERR_ARG;
    if (!maps[l].drows || !maps[l].rows || !maps[l].inv) return PNCE_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(maps[l].drows) & 15u) || (reinterpret_cast<uintptr_t>(maps[l].rows) & 15u)) return PNCE_ERR_ALIGN;
    if (maps[l].dfeat == nullptr) dense = false;                // maps without gradient: every dfeat NULL
    else if (reinterpret_cast<uintptr_t>(maps[l].dfeat) & (dtype_size(dtype) - 1)) return PNCE_ERR_ALIGN;
  }
  if (!dense)
    for (int l = 0; l < n_maps; ++l)
      if (maps[l].dfeat != nullptr) return PNCE_ERR_ARG;
  pg.dtype = dtype;
  pg.math = math_mode;
  pg.nhwc = layout == PNCE_LAYOUT_NHWC ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // 1. normalise backward, d loss / d Y as a row blob
  {
    static thread_local NetfPackLaunch pk;
    memset(&pk, 0, sizeof(pk));
    pk.n = n_maps; pk.B = batch;
    long long acc = 0;
    for (int l = 0; l < n_maps; ++l) {
      const LayerDev& G = pg.L[l];
      NetfPackJob& j = pk.job[l];
      j.g = maps[l].drows; j.y = maps[l].rows; j.inv = maps[l].inv; j.perm = G.perm;
      j.hi = np.dy[l][0]; j.lo = np.dy[l][1];
      j.P = G.P; j.Ppad = G.Ppad; j.N = nc;
      pk.start[l] = acc;
      acc += ((long long)batch * G.Ppad + 7) / 8;
    }
    pk.start[n_maps] = acc;
    if (acc > 0x7fffffffLL) return PNCE_ERR_UNSUPPORTED;
    launch_k(k_netf_dy_pack, (unsigned)acc, kThreads, 0, st, pk);
    PNCE_CUDA(cudaGetLastError());
  }
  // 2. dH = (dY W2) * [H > 0]
  static thread_local GemmLaunch g;
  memset(&g, 0, sizeof(g));
  g.x3 = x3 ? 1 : 0;
  g.err = dev_status;
  for (int l = 0; l < n_maps; ++l) {
    const HeadLayerBufs& hb = np.hb[l];
    const LayerDev& G = pg.L[l];
    GemmProb& pr = g.pr[g.n++];
    pr.a_hi = np.dy[l][0]; pr.a_lo = np.dy[l][1]; pr.b_hi = hb.w2t[0]; pr.b_lo = hb.w2t[1];
    pr.K = nc; pr.N = nc; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_DH;
    pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = nc;
    pr.o_hi = hb.dh[0]; pr.o_lo = hb.dh[1]; pr.mask_hi = hb.hq[0];
  }
  rc = launch_gemm(g, st);
  if (rc != PNCE_OK) return rc;
  // 3. dX = dH W1 -> the gradient rows the dense backward reads
  if (dense) {
    memset(&g, 0, sizeof(g));
    g.x3 = x3 ? 1 : 0;
    g.err = dev_status;
    for (int l = 0; l < n_maps; ++l) {
      const HeadLayerBufs& hb = np.hb[l];
      const LayerDev& G = pg.L[l];
      GemmProb& pr = g.pr[g.n++];
      pr.a_hi = hb.dh[0]; pr.a_lo = hb.dh[1]; pr.b_hi = hb.w1t[0]; pr.b_lo = hb.w1t[1];
      pr.K = nc; pr.N = G.Cp; pr.tiles = batch * (G.Ppad / 128); pr.mode = GM_DX;
      pr.P = G.P; pr.Ppad = G.Ppad; pr.halves = G.Ppad / 128; pr.C = G.C;
      pr.outT = G.dxT; pr.rm = pg.nhwc;
    }
    rc = launch_gemm(g, st);
    if (rc != PNCE_OK) return rc;
  }
  // 4. weight / bias gradients (split-K partials + deterministic reduce)
  static thread_local WgradLaunch wg;
  memset(&wg, 0, sizeof(wg));
  wg.x3 = x3 ? 1 : 0;
  wg.err = dev_status;
  long long acc = 0;
  for (int l = 0; l < n_maps; ++l) {
    const HeadLayerBufs& hb = np.hb[l];
    const LayerDev& G = pg.L[l];
    const int tiles = batch * (G.Ppad / 128);
    for (int which = 0; which < 2; ++which) {
      WgradProb& pr = wg.pr[wg.n];
      pr.a_hi = which ? hb.dh[0] : np.dy[l][0]; pr.a_lo = which ? hb.dh[1] : np.dy[l][1];
      pr.b_hi = which ? hb.xq[0] : hb.hq[0]; pr.b_lo = which ? hb.xq[1] : hb.hq[1];
      pr.NA = nc; pr.N = which ? G.Cp : nc; pr.tiles = tiles; pr.slabs = hb.slabs;
      pr.partial = which ? hb.pw1 : hb.pw2; pr.pbias = which ? hb.pb1 : hb.pb2;
      wg.start[wg.n++] = acc;
      acc += (long long)hb.slabs * (nc / 128);
    }
  }
  wg.start[wg.n] = acc;
  rc = set_smem(k_wgrad_tc, kWgSmemBytes);
  if (rc != PNCE_OK) return rc;
  launch_k(k_wgrad_tc, (unsigned)acc, kTcThreads, kWgSmemBytes, st, wg);
  PNCE_CUDA(cudaGetLastError());
  {
    static thread_local WreduceLaunch rl;
    memset(&rl, 0, sizeof(rl));
    rl.grad_out = nullptr;                                     // the incoming rows already carry the upstream gradient
    int blocks = 0;
    for (int l = 0; l < n_maps; ++l) {
      const HeadLayerBufs& hb = np.hb[l];
      const LayerDev& G = pg.L[l];
      for (int which = 0; which < 2; ++which) {
        WreduceJob& j = rl.job[rl.n];
        j.partial = which ? hb.pw1 : hb.pw2; j.pbias = which ? hb.pb1 : hb.pb2;
        j.dw = which ? heads[l].dw1 : heads[l].dw2; j.db = which ? heads[l].db1 : heads[l].db2;
        j.NA = nc; j.N = which ? G.Cp : nc; j.Nout = which ? G.C : nc; j.slabs = hb.slabs;
        rl.start[rl.n++] = blocks;
        blocks += (int)(((long long)nc * j.N + nc + kThreads - 1) / kThreads);
      }
    }
    rl.start[rl.n] = blocks;
    launch_k(k_wreduce, (unsigned)blocks, kThreads, 0, st, rl);
    PNCE_CUDA(cudaGetLastError());
  }
  // 5. dense d feat (zero fill + sampled positions)
  if (!dense) return PNCE_OK;
  pg.grad_out = nullptr;
  return launch_dense(pg, st);
}

int pnce_multi_axpby(float* const* dev_dst, const float* const* dev_src, const long long* dev_numel,
                     const int* dev_chunk_tensor, const long long* dev_chunk_start, int n_chunks, float a, float b,
                     int mode, void* stream) {
  if (!dev_dst || !dev_src || !dev_numel || !dev_chunk_tensor || !dev_chunk_start || n_chunks < 0) return PNCE_ERR_ARG;
  if (mode != 0 && mode != 1) return PNCE_ERR_ARG;
  if (n_chunks == 0) return PNCE_OK;
  launch_k(k_multi_axpby, (unsigned)n_chunks, kMtThreads, 0, static_cast<cudaStream_t>(stream), 
      dev_dst, dev_src, dev_numel, dev_chunk_tensor, dev_chunk_start, a, b, mode);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}
int pnce_multi_chunk_elems(void) { return kMtChunk; }

int pnce_amp_adam_step(float* const* dev_param, float* const* dev_grad, float* const* dev_exp_avg,
                       float* const* dev_exp_avg_sq, float* const* dev_step, const long long* dev_numel,
                       const int* dev_chunk_tensor, const long long* dev_chunk_start, int n_chunks, int n_tensors,
                       float* dev_scale, int* dev_growth_tracker, float growth_factor, float backoff_factor,
                       int growth_interval, float max_grad_norm, double lr, double beta1, double beta2, double eps,
                       double weight_decay, float* dev_scratch, void* stream) {
  if (!dev_param || !dev_grad || !dev_exp_avg || !dev_exp_avg_sq || !dev_step || !dev_numel || !dev_chunk_tensor ||
      !dev_chunk_start || !dev_scratch || n_chunks < 0 || n_tensors < 0)
    return PNCE_ERR_ARG;
  if ((dev_scale == nullptr) != (dev_growth_tracker == nullptr)) return PNCE_ERR_ARG;
  if (dev_scale && growth_interval < 1) return PNCE_ERR_ARG;
  if (!(lr >= 0.0) || !(beta1 >= 0.0 && beta1 < 1.0) || !(beta2 >= 0.0 && beta2 < 1.0) || !(eps >= 0.0) ||
      !(weight_decay >= 0.0))
    return PNCE_ERR_ARG;                                         // the checks of torch.optim.Adam.__init__
  AmpAdamTable a;
  a.param = dev_param; a.grad = dev_grad; a.m = dev_exp_avg; a.v = dev_exp_avg_sq; a.step = dev_step;
  a.numel = dev_numel; a.chunk_tensor = dev_chunk_tensor; a.chunk_start = dev_chunk_start;
  a.n_chunks = n_chunks; a.n_tensors = n_tensors;
  a.scale = dev_scale; a.growth_tracker = dev_growth_tracker;
  a.growth_factor = growth_factor; a.backoff_factor = backoff_factor; a.growth_interval = growth_interval;
  a.max_norm = max_grad_norm;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
  a.scratch = dev_scratch;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_chunks > 0) {
    launch_k(k_amp_gradnorm, (unsigned)n_chunks, kMtThreads, 0, st, a);
    launch_k(k_amp_adam, (unsigned)n_chunks, kMtThreads, 0, st, a);
  }
  launch_k(k_amp_finish, 1, kMtThreads, 0, st, a);       // with no gradients at all GradScaler.update() still runs
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}
// ---- D-side row (SURVEY.md section 8f row 4) -------------------------------------------------------------------
static int aug_blocks(int H, int W) {
  const int per = (H * W + kAugThreads - 1) / kAugThreads;
  return per < 32 ? per : 32;
}
size_t pnce_diffaug_scratch_floats(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)B * aug_blocks(H, W);
}
int pnce_diffaug(const void* dev_in, void* dev_out, int dtype, int B, int C, int H, int W, const void* dev_rb,
                 const void* dev_rs, const void* dev_rc, const long long* dev_tx, const long long* dev_ty,
                 const long long* dev_ox, const long long* dev_oy, int cut_h, int cut_w, float* dev_scratch,
                 int backward, void* stream) {
  if (!dev_in || !dev_out || dev_in == dev_out || B <= 0 || C <= 0 || H <= 0 || W <= 0) return PNCE_ERR_ARG;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (C > kAugMaxC || (long long)C * H * W > 0x7fffffffLL || B > 65535) return PNCE_ERR_UNSUPPORTED;
  const bool color = dev_rb != nullptr;
  if (color != (dev_rs != nullptr) || color != (dev_rc != nullptr)) return PNCE_ERR_ARG;   // 'color' is all three
  if ((dev_tx != nullptr) != (dev_ty != nullptr)) return PNCE_ERR_ARG;
  const bool cut = cut_h > 0 || cut_w > 0;
  if (cut && (cut_h <= 0 || cut_w <= 0 || !dev_ox || !dev_oy)) return PNCE_ERR_ARG;
  if (color && !dev_scratch) return PNCE_ERR_WORKSPACE;
  AugParams a;
  memset(&a, 0, sizeof(a));
  a.x = dev_in; a.y = dev_out; a.dtype = dtype; a.B = B; a.C = C; a.H = H; a.W = W;
  a.rb = dev_rb; a.rs = dev_rs; a.rc = dev_rc; a.tx = dev_tx; a.ty = dev_ty;
  a.ox = cut ? dev_ox : nullptr; a.oy = cut ? dev_oy : nullptr;
  a.cut_h = cut ? cut_h : 0; a.cut_w = cut ? cut_w : 0;
  a.part = dev_scratch; a.nblk = aug_blocks(H, W);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 rgrid((unsigned)a.nblk, (unsigned)B), grid((unsigned)((H * W + kAugThreads - 1) / kAugThreads), (unsigned)B);
#define PNCE_AUG_LAUNCH(T)                                                              \
  do {                                                                                  \
    if (color) {                                                                        \
      if (backward) launch_k(k_aug_reduce<T, true>, rgrid, kAugThreads, 0, st, a);            \
      else launch_k(k_aug_reduce<T, false>, rgrid, kAugThreads, 0, st, a);                    \
    }                                                                                   \
    if (backward) launch_k(k_aug_bwd<T>, grid, kAugThreads, 0, st, a);                        \
    else launch_k(k_aug_fwd<T>, grid, kAugThreads, 0, st, a);                                 \
  } while (0)
  if (dtype == PNCE_F32) PNCE_AUG_LAUNCH(float);
  else if (dtype == PNCE_F16) PNCE_AUG_LAUNCH(__half);
  else PNCE_AUG_LAUNCH(__nv_bfloat16);
#undef PNCE_AUG_LAUNCH
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

static int hinge_fill(HingeParams& h, const void* const* real, const void* const* fake, void* const* dreal,
                      void* const* dfake, const long long* numel, int scales, int mode, int dtype) {
  if (!fake || !numel || scales < 1 || (mode != 0 && mode != 1)) return PNCE_ERR_ARG;
  if (scales > kHingeMaxScales) return PNCE_ERR_UNSUPPORTED;
  if (dtype < PNCE_F32 || dtype > PNCE_BF16) return PNCE_ERR_ARG;
  if (mode == 0 && !real) return PNCE_ERR_ARG;
  memset(&h, 0, sizeof(h));
  for (int s = 0; s < scales; ++s) {
    if (!fake[s] || (mode == 0 && !real[s]) || numel[s] <= 0) return PNCE_ERR_ARG;
    h.fake[s] = fake[s];
    h.real[s] = mode == 0 ? real[s] : nullptr;
    h.dreal[s] = dreal ? dreal[s] : nullptr;
    h.dfake[s] = dfake ? dfake[s] : nullptr;
    h.n[s] = numel[s];
  }
  h.scales = scales; h.mode = mode; h.dtype = dtype;
  return PNCE_OK;
}
int pnce_hinge_fwd(const void* const* real, const void* const* fake, const long long* numel, int scales, int mode,
                   int dtype, float* dev_loss, void* stream) {
  HingeParams h;
  int rc = hinge_fill(h, real, fake, nullptr, nullptr, numel, scales, mode, dtype);
  if (rc != PNCE_OK) return rc;
  if (!dev_loss) return PNCE_ERR_ARG;
  h.loss = dev_loss;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == PNCE_F32) launch_k(k_hinge_fwd<float>, 1, kAugThreads, 0, st, h);
  else if (dtype == PNCE_F16) launch_k(k_hinge_fwd<__half>, 1, kAugThreads, 0, st, h);
  else launch_k(k_hinge_fwd<__nv_bfloat16>, 1, kAugThreads, 0, st, h);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}
int pnce_hinge_bwd(const void* const* real, const void* const* fake, void* const* dreal, void* const* dfake,
                   const long long* numel, int scales, int mode, int dtype, const float* dev_grad_out, void* stream) {
  HingeParams h;
  int rc = hinge_fill(h, real, fake, dreal, dfake, numel, scales, mode, dtype);
  if (rc != PNCE_OK) return rc;
  if (!dev_grad_out) return PNCE_ERR_ARG;
  h.grad_out = dev_grad_out;
  long long mx = 0;
  for (int s = 0; s < scales; ++s) mx = numel[s] > mx ? numel[s] : mx;
  long long gx = (mx + kAugThreads - 1) / kAugThreads;
  if (gx > 1024) gx = 1024;
  const dim3 grid((unsigned)gx, (unsigned)scales);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == PNCE_F32) launch_k(k_hinge_bwd<float>, grid, kAugThreads, 0, st, h);
  else if (dtype == PNCE_F16) launch_k(k_hinge_bwd<__half>, grid, kAugThreads, 0, st, h);
  else launch_k(k_hinge_bwd<__nv_bfloat16>, grid, kAugThreads, 0, st, h);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

size_t pnce_amp_adam_scratch_floats(int n_chunks) { return (size_t)(n_chunks < 0 ? 0 : n_chunks) + 2; }

int pnce_selftest_umma(const void* a_blob, size_t a_bytes, const void* b_blob, size_t b_bytes,
                       unsigned a_lbo, unsigned a_sbo, unsigned a_kstep, unsigned b_lbo, unsigned b_sbo,
                       unsigned b_kstep, int n, int k, int b_mn_major, float* d_out, int* err, void* stream) {
  if (!a_blob || !b_blob || !d_out || !err) return PNCE_ERR_ARG;
  if (n < 16 || n > 256 || (n % 32) || k < 16 || (k % 16) || (a_bytes % 16) || (b_bytes % 16)) return PNCE_ERR_ARG;
  ProbeArgs a;
  a.a_blob = a_blob; a.b_blob = b_blob; a.d_out = d_out; a.err = err;
  a.a_bytes = (uint32_t)a_bytes; a.b_bytes = (uint32_t)b_bytes;
  a.a_lbo = a_lbo; a.a_sbo = a_sbo; a.a_kstep = a_kstep;
  a.b_lbo = b_lbo; a.b_sbo = b_sbo; a.b_kstep = b_kstep;
  a.n = n; a.k = k; a.b_mn_major = b_mn_major;
  const size_t smem = ((a_bytes + 1023) & ~(size_t)1023) + b_bytes;
  int rc = set_smem(k_umma_probe, smem);
  if (rc != PNCE_OK) return rc;
  k_umma_probe<<<1, 128, smem, static_cast<cudaStream_t>(stream)>>>(a);
  PNCE_CUDA(cudaGetLastError());
  return PNCE_OK;
}

}  // extern "C"
