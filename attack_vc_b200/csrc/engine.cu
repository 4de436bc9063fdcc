// engine.cu -- host side of libavc_b200.so: handle, weight packing, launch plans for the three
// attacks (attack_utils.py:7-130) and the C-ABI declared in include/avc_b200.h.
//
// A "plan" is the ordered list of kernel launches of one attack iteration for fixed shapes.  It is
// built once, captured into a CUDA graph and replayed n_iters times; nothing in the loop touches the
// host (the reference never reads the loss inside the loop either, SURVEY §3.1).
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/avc_b200.h"
#include "host_util.h"
#include "conv_simt.cuh"
#include "conv_tc.cuh"
#include "conv_tc2.cuh"
#include "conv_wgrad.cuh"
#include "wgrad_tc.cuh"
#include "conv2d_tc.cuh"
#include "elementwise.cuh"

using namespace avc;

namespace {

thread_local std::string g_create_error;

// Every kernel of the loop is launched with programmatic dependent launch (PDL): the next kernel's
// CTAs may become resident while the previous kernel drains, run their data-independent prologue
// (weight prefetch) and block in griddepcontrol.wait until the predecessor's memory is visible.
bool g_pdl = getenv("AVC_NO_PDL") == nullptr;
template <class... KArgs, class... Args>
void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = g_pdl ? 1 : 0;
  CK(cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...));
}
// the same as a grid of clusters of `csize` CTAs (2: CTA pairs on one TPC for the tcgen05 cta_group::2 kernel)
template <class... KArgs, class... Args>
void launch_k_cluster(unsigned csize, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = csize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = g_pdl ? 2 : 1;
  CK(cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...));
}

// ---- packed weights ----------------------------------------------------------------------------
struct ConvW {
  int c_in = 0, c_out = 0, k = 0, stride = 1;
  float* fwd = nullptr;   // [k][c_in][c_out']      c_out' = pixel-shuffle-permuted output channel
  float* bwd = nullptr;   // [k reversed][c_out'][c_in]
  float* bias = nullptr;  // [c_out']
  TcPack tc_fwd[4], tc_bwd[4];  // tcgen05 operand images per tap residue mod stride (conv_tc.cuh); !ok when not eligible
  float *fwd_h = nullptr, *fwd_l = nullptr;   // hi / lo planes of fwd (1x1 convs only): the K-major weight operand of the TMA-fed dgrad (conv2d_tc.cuh)
  int pl() const { return k / 2; }
  int pr() const { return (k % 2) ? k / 2 : k / 2 - 1; }
};


// Tensor-core view of one plain Conv1d (any stride), forward or dgrad -- see conv_tc.cuh.
//   forward: one group per tap residue e (taps j = s*i + e read input position s*(t+i) + e - pl)
//   dgrad:   one pass per output residue e (rows p = s*u + e of the padded gradient use taps j = s*i + e)
// N > 128 is split into passes of 128 columns.
TcOp tc_op_conv(const ConvW& w, bool bwd) {
  TcOp op;
  const int s = w.stride;
  if (s > 4) return TcOp{};
  if (!bwd) {
    op.n_out = w.c_out;
    for (int e = 0; e < s && e < w.k; ++e) if (!w.tc_fwd[e].ok) return TcOp{};
    const int nch = w.tc_fwd[0].n_chunks;
    for (int ch = 0; ch < nch; ++ch) {
      const int g0 = op.n_groups;
      for (int e = 0; e < s && e < w.k; ++e)
        if (op.add_group(w.tc_fwd[e].blocks[ch], 0, w.c_in, w.tc_fwd[e].k, s, e - w.pl()) < 0) return TcOp{};
      if (!op.add_pass(g0, op.n_groups, w.tc_fwd[0].cn[ch], ch * kTcNMax, 1, 0)) return TcOp{};
    }
  } else {
    op.n_out = w.c_in;
    op.sdiv = s;
    for (int e = 0; e < s && e < w.k; ++e) if (!w.tc_bwd[e].ok) return TcOp{};
    const int nch = w.tc_bwd[0].n_chunks;
    for (int e = 0; e < s && e < w.k; ++e)
      for (int ch = 0; ch < nch; ++ch) {
        const int g0 = op.add_group(w.tc_bwd[e].blocks[ch], 0, w.c_out, w.tc_bwd[e].k, 1, -(w.tc_bwd[e].k - 1));
        if (g0 < 0 || !op.add_pass(g0, g0 + 1, w.tc_bwd[e].cn[ch], ch * kTcNMax, s, e - w.pl())) return TcOp{};
      }
  }
  return op;
}


// f: forward image [k][c_in][c_out'], r: dgrad image [k reversed][c_out'][c_in] (pack_conv)
void tc_pack_both(Arena& mem, ConvW& c, const std::vector<float>& f, const std::vector<float>& r) {
  const int s = c.stride, k = c.k;
  for (int e = 0; e < s && e < k && e < 4; ++e) {
    std::vector<int> ft, bt;
    for (int j = e; j < k; j += s) ft.push_back(j);                 // window order = ascending tap
    const int ne = (int)ft.size();
    for (int tp = 0; tp < ne; ++tp) bt.push_back(k - 1 - (s * (ne - 1 - tp) + e));   // image index of W_j^T, j = s*(ne-1-tp)+e
    tc_pack_taps(mem, c.tc_fwd[e], f, c.c_in, c.c_out, ft);
    tc_pack_taps(mem, c.tc_bwd[e], r, c.c_out, c.c_in, bt);
  }
}

struct EncoderW {
  avc_encoder_desc d{};
  int n_bank = 0, c_cat = 0;
  ConvW bank[AVC_MAX_BANK];
  float* bank_bias = nullptr;   // [n_bank*c_bank]
  ConvW in_conv, c1[AVC_MAX_BLOCKS], c2[AVC_MAX_BLOCKS];
  ConvW mean_layer;             // content encoder only
  // dense tail (speaker encoder only)
  float *Wt1[AVC_MAX_BLOCKS]{}, *Wt2[AVC_MAX_BLOCKS]{}, *W1[AVC_MAX_BLOCKS]{}, *W2[AVC_MAX_BLOCKS]{}, *b1[AVC_MAX_BLOCKS]{}, *b2[AVC_MAX_BLOCKS]{};
  float *Wto = nullptr, *Wo = nullptr, *bo = nullptr;
};

struct DecoderW {
  avc_decoder_desc d{};
  ConvW in_conv, c1[AVC_MAX_BLOCKS], c2[AVC_MAX_BLOCKS], out_conv;
  float *aWt[2 * AVC_MAX_BLOCKS]{}, *aW[2 * AVC_MAX_BLOCKS]{}, *ab[2 * AVC_MAX_BLOCKS]{};
};

enum LaunchKind : int { LK_CONV = 0, LK_NORM = 1, LK_TAIL = 2, LK_AFFINE = 3, LK_LOSS = 4, LK_UPDATE = 5, LK_LAYOUT = 6, LK_COPY = 7 };

struct Launch {
  std::function<void(cudaStream_t)> fn;
  int kind = LK_COPY;
  double flops = 0;   // algorithmic FLOPs of this launch (2 per MAC; dgrad of a strided conv counts real taps only)
  double bytes = 0;   // algorithmic HBM bytes (each tensor touched once)
  void operator()(cudaStream_t st) const { fn(st); }
};

constexpr int kUnroll = 16;

// Caller tensors of one attack call.  Setup / finish launches read them through the plan at LAUNCH time, so a cached
// plan (same shapes, eps, normaliser) is rebound to the next call's tensors without rebuilding or re-capturing.
struct IoBind {
  const float* vc_tgt = nullptr;  int64_t tgt_stride[3] = {0, 0, 0};
  const float* adv_tgt = nullptr; int64_t adv_stride[3] = {0, 0, 0};
  const float* vc_src = nullptr;  int64_t src_stride[3] = {0, 0, 0};
  const float* w0 = nullptr;      int64_t w0_stride[3] = {0, 0, 0};
  float* adv_out = nullptr;       int64_t out_stride[3] = {0, 0, 0};
  float* loss_out = nullptr;
  float* grad_out = nullptr;
  int n_iters = 0;                 // iterations of THIS call (<= Plan::n_iters, the provisioned capacity)
  void bind(const avc_attack_args& a) {
    vc_tgt = a.vc_tgt; adv_tgt = a.adv_tgt; vc_src = a.vc_src; w0 = a.w0; adv_out = a.adv_out;
    loss_out = a.loss_out; grad_out = a.grad_out; n_iters = a.n_iters;
    for (int i = 0; i < 3; ++i) {
      tgt_stride[i] = a.tgt_stride[i]; adv_stride[i] = a.adv_stride[i]; src_stride[i] = a.src_stride[i];
      w0_stride[i] = a.w0_stride[i]; out_stride[i] = a.out_stride[i];
    }
  }
};

struct PlanKey {
  int kind = -1, B = 0, T_tgt = 0, T_adv = 0, T_src = 0, use_graph = 0, has_grad = 0, conv_impl = 0;
  long long tc_min_rows = 0;
  float eps = 0.f;
  double inv_norm = 0.0;
  std::vector<int> frames;   // ragged plans: every utterance's length (empty: equal lengths)
  bool operator==(const PlanKey& o) const {
    return kind == o.kind && B == o.B && T_tgt == o.T_tgt && T_adv == o.T_adv && T_src == o.T_src && use_graph == o.use_graph &&
           has_grad == o.has_grad && conv_impl == o.conv_impl && tc_min_rows == o.tc_min_rows && eps == o.eps && inv_norm == o.inv_norm &&
           frames == o.frames;
  }
};

struct Plan {
  Arena mem;
  IoBind io;
  PlanKey key;
  Plan(SlabPool* pool, cudaStream_t st) : mem(pool, st) {}
  std::vector<Launch> setup;    // once per attack call (targets, loop invariants)
  std::vector<Launch> iter;     // one attack iteration
  std::vector<Launch> iter2;    // header optimisation only: the apply half of an iteration (after the gradient all-reduce)
  float* gh = nullptr; long long gh_n = 0;   // header optimisation: this rank's partial gradient [T,C]
  std::vector<Launch> finish;   // after the loop
  cudaGraph_t graph = nullptr, graphU = nullptr;
  cudaGraphExec_t exec = nullptr;    // one iteration
  cudaGraphExec_t execU = nullptr;   // kUnroll iterations back to back: 16x fewer launches, shallow launch queue
  cudaGraph_t graph2 = nullptr; cudaGraphExec_t exec2 = nullptr;   // header optimisation: apply half
  int n_iters = 0;      // iterations the Adam table / loss buffer were sized for
  int done_iters = 0;
  bool use_graph = true;
  bool finished = false;
  ~Plan() {
    if (exec) cudaGraphExecDestroy(exec);
    if (execU) cudaGraphExecDestroy(execU);
    if (exec2) cudaGraphExecDestroy(exec2);
    if (graph2) cudaGraphDestroy(graph2);
    if (graph) cudaGraphDestroy(graph);
    if (graphU) cudaGraphDestroy(graphU);
  }
};

}  // namespace

struct avc_handle {
  int device = 0;
  int sm_count = 148;
  avc_model_desc desc{};
  Arena wmem;
  SlabPool pool;      // activation slabs recycled between attacks (declared before any Plan can die)
  bool have_weights = false;
  EncoderW se, ce;
  DecoderW dec;
  std::string err;
  long long launches = 0;
  int launches_per_iter = 0;
  int conv_impl = 0;   // 0 auto, 1 fp32 CUDA cores, 2 tcgen05 (TF32 + BF16 correction), 3 CUDA cores without the small-M kernel, 4 tcgen05 single TF32 pass (measurement only),
                       // 6 tcgen05 with the role-swapped N = 256 kernel forced, 7 tcgen05 with the N = 128 kernel forced
  long long tc_min_rows = 2048;   // auto: GEMM rows from which the tensor-core kernel is used (env AVC_TC_MIN_ROWS)
  // Finished attack plans (buffers, launch lists, instantiated graphs) kept for the next call of the same shape: building
  // and capturing a plan costs ~1 ms, as much as a few iterations at batch 1.  Small plans only, a handful of them.
  std::vector<std::unique_ptr<Plan>> plan_cache;
  long long plan_cache_hits = 0;
  // avc_unit_timing: the HBM-bound unit entry points run their launch list 1 + unit_reps times back to back and time the
  // last unit_reps with events recorded on the caller's stream right behind the first run (no host time in the bracket)
  int unit_reps = 0;
  float unit_ms = 0.f;
};

struct avc_session {
  avc_handle* h;
  std::unique_ptr<Plan> plan;
};

namespace {

// =================================================================================================
// conv launch
// =================================================================================================
constexpr size_t kSmemMax = 227 * 1024;

template <int RM, int TXN, int TYN>
void launch_conv_cfg(ConvArgs a, cudaStream_t st) {
  constexpr int TM = RM * TYN, TN = TXN * 4;
  a.win_rows = a.bwd ? TM + 16 : (TM - 1) * a.s + kMaxTaps;
  const size_t smem = ((size_t)(a.win_rows + kMaxTaps) * kSRow + 2 * kKSub * TN) * sizeof(float);
  if (smem > 200 * 1024) fail(AVC_ERR_INVALID, "conv window needs %zu B of shared memory", smem);
  const int tiles_t = (a.T_y + TM - 1) / TM;
  dim3 grid(a.B * tiles_t, (a.N + TN - 1) / TN, a.zsplit ? a.n_groups : 1);
  launch_k(conv_simt_kernel<RM, TXN, TYN>, grid, TXN * TYN, smem, st, a);
}

void init_kernel_attributes() {
  wt_init_attributes();
  c2_init_attributes();
  CK(cudaFuncSetAttribute(conv_simt_kernel<4, 16, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(conv_simt_kernel<2, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(conv_simt_kernel<1, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(conv_small_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CK(cudaFuncSetAttribute(conv_small_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  constexpr int tcl_smem = 2 * (2 * kTailMaxDense + 1) * kTclMatBytes > (int)kSmemMax - 4096 ? (int)kSmemMax - 4096 : 2 * (2 * kTailMaxDense + 1) * kTclMatBytes;
  CK(cudaFuncSetAttribute(se_tail_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmem));
  CK(cudaFuncSetAttribute(se_tail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmem));
  CK(cudaFuncSetAttribute(se_tail_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tcl_smem));
  CK(cudaFuncSetAttribute(se_tail_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tcl_smem));
  CK(cudaFuncSetAttribute(norm_act_fwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(norm_act_fwd_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(norm_act_fwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(norm_act_bwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(norm_act_bwd_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(norm_act_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kNormSmemMax));
  CK(cudaFuncSetAttribute(conv_tc_kernel_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CK(cudaFuncSetAttribute(conv_tc_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CK(cudaFuncSetAttribute(conv_tc_kernel_t<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CK(cudaFuncSetAttribute(conv_tc2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CK(cudaFuncSetAttribute(conv_tc2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
}

// small-M path: every window resident, deep weight ring (conv_simt.cuh: conv_small_kernel)
template <int TM>
bool small_cfg(ConvArgs& a, dim3& grid, size_t& smem) {
  const int tiles_t = (a.T_y + TM - 1) / TM;
  int rows[kMaxGroups] = {0}, kc_max = 0, slabs_max = 0, slabs_all = 0;
  for (int g = 0; g < a.n_groups; ++g) {
    for (int i = 0; i < tiles_t; ++i) {
      const WinGeom w = win_geom(a.bwd, a.s, a.T_y, a.g[g], i * TM, std::min(i * TM + TM, a.T_y));
      rows[g] = std::max(rows[g], w.nrows);
    }
    if (a.g[g].kc % kSmKW) return false;   // the kernel gives every warp a whole K slice
    kc_max = std::max(kc_max, a.g[g].kc);
    slabs_max = std::max(slabs_max, a.g[g].n_taps);
    slabs_all += a.g[g].n_taps;
  }
  // window rows: every group of a CTA is resident at once; with a z split (conv bank forward: one group per z; K split:
  // a range of groups per z) the offsets restart for every z and the region is sized for the largest
  const int n_rng = a.zk > 1 ? a.zk : 1;
  int off = 0, slabs_rng = 0;
  for (int r = 0; r < n_rng; ++r) {
    const int lo = a.zk > 1 ? a.zk_lo[r] : 0, hi = a.zk > 1 ? a.zk_hi[r] : a.n_groups;
    int o = 0, sl = 0;
    for (int g = lo; g < hi; ++g) {
      a.win_off[g] = a.zsplit ? 0 : o;
      o = a.zsplit ? std::max(o, rows[g]) : o + rows[g];
      sl += a.g[g].n_taps;
    }
    off = std::max(off, o);
    slabs_rng = std::max(slabs_rng, sl);
  }
  a.win_off[a.n_groups] = off;
  a.slab_floats = kc_max * kSmTN;
  // dgrad: rows for the pre-summed operands of reflect-edge output rows (conv_small_kernel); skipped when a tile's left and
  // right border rows overlap (tiny T) or the rows would take too much shared memory -- the kernel then sums inside the loop
  a.e_rows = 0;
  static const bool no_edge_pre = getenv("AVC_NO_EDGE_PRE") != nullptr;
  if (a.bwd && !a.zsplit && !no_edge_pre) {
    int e_max = 0; bool ok = true;
    for (int r = 0; r < n_rng && ok; ++r) {
      const int lo = a.zk > 1 ? a.zk_lo[r] : 0, hi = a.zk > 1 ? a.zk_hi[r] : a.n_groups;
      int e_tot = 0;
      for (int g = lo; g < hi && ok; ++g) {
        int need = 0;
        for (int i = 0; i < tiles_t; ++i) {
          const WinGeom w = win_geom(a.bwd, a.s, a.T_y, a.g[g], i * TM, std::min(i * TM + TM, a.T_y));
          const int nl = std::max(0, w.lt_hi - w.lt_lo + 1), nr = std::max(0, w.rt_hi - w.rt_lo + 1);
          if (nl && nr && w.lt_hi >= w.rt_lo) ok = false;
          need = std::max(need, (nl + nr) * a.g[g].n_taps);
        }
        a.e_off[g] = off + kMaxTaps + e_tot;
        e_tot += need;
      }
      e_max = std::max(e_max, e_tot);
    }
    if (ok && e_max > 0 && (size_t)e_max * kSRow * sizeof(float) <= 56 * 1024) a.e_rows = e_max;
  }
  const size_t win_bytes = (size_t)(off + kMaxTaps + a.e_rows) * kSRow * sizeof(float);
  const size_t slab_bytes = (size_t)a.slab_floats * sizeof(float);
  // fold regions behind the ring: constants | staged partials | second-operand window | epilogue operands
  size_t fold_floats = 0;
  a.f_stage = a.f_s2 = a.f_epi = 0;
  if (a.pro.mode) {
    a.f_stage = kFoldPC;
    a.f_s2 = a.f_stage + a.pro.n_part * a.pro.C * 2;
    const bool second = a.pro.mode == 2 || a.pro.res.mode != RES_NONE;
    fold_floats = (size_t)a.f_s2 + (second ? (size_t)off * kSRow : 0);
  }
  if (a.epi.mode == 2) { a.f_epi = (int)fold_floats; fold_floats += (size_t)TM * kSmTN + 128; }
  const size_t fold_bytes = fold_floats * sizeof(float);
  const size_t avail = kSmemMax - fold_bytes;
  const int n_slabs = a.zsplit ? slabs_max : a.zk > 1 ? slabs_rng : slabs_all;
  if (win_bytes + 2 * slab_bytes > avail) return false;
  // a ring that holds every slab (n_slabs + 1 buffers) needs no refills and no per-slab barrier; else at most 8 buffers
  int ring = (int)((avail - win_bytes) / slab_bytes);
  if (ring < n_slabs) ring = std::min(ring, 8);
  ring = std::max(2, std::min(ring, n_slabs));
  while ((size_t)ring * slab_bytes < (size_t)kSmWarps * TM * kSmTN * sizeof(float)) ++ring;   // the ring doubles as the split-K reduction buffer
  smem = win_bytes + (size_t)ring * slab_bytes + fold_bytes;
  if (smem > kSmemMax) return false;
  a.ring = ring;
  grid = dim3(a.B * tiles_t, (a.N + kSmTN - 1) / kSmTN, a.zsplit ? a.n_groups : a.zk > 1 ? a.zk : 1);
  return true;
}
template <int TM>
bool launch_conv_small_cfg(ConvArgs a, cudaStream_t st) {
  dim3 grid; size_t smem = 0;
  if (!small_cfg<TM>(a, grid, smem)) return false;
  launch_k(conv_small_kernel<TM>, grid, 32 * kSmWarps, smem, st, a);
  return true;
}

// tile height the small-M kernel would run this conv with; 0: one of the generic tiles takes it
int small_tm(const ConvArgs& a, int sm_count, bool allow_small = true) {
  const long long z = a.zsplit ? a.n_groups : a.zk > 1 ? a.zk : 1;
  auto ctas = [&](int TM, int TN) { return (long long)a.B * ((a.T_y + TM - 1) / TM) * ((a.N + TN - 1) / TN) * z; };
  if (ctas(64, 64) >= 2LL * sm_count || ctas(32, 32) >= 2LL * sm_count) return 0;
  static const bool no_small = getenv("AVC_NO_SMALL") != nullptr;
  if (no_small || !allow_small) return 0;
  ConvArgs t = a; dim3 g; size_t sm = 0;
  if (ctas(8, kSmTN) <= sm_count) return small_cfg<8>(t, g, sm) ? 8 : 0;
  return small_cfg<16>(t, g, sm) ? 16 : 0;
}

void launch_conv_simt(const ConvArgs& a, int sm_count, cudaStream_t st, bool allow_small = true) {
  // pick the largest tile that still gives every SM about two CTAs; small-M problems (batch 1)
  // take the latency-oriented kernel
  const int tm = small_tm(a, sm_count, allow_small);
  if (tm == 8 && launch_conv_small_cfg<8>(a, st)) return;
  if (tm == 16 && launch_conv_small_cfg<16>(a, st)) return;
  if (a.pro.mode || a.epi.mode || a.zk > 1) fail(AVC_ERR_STATE, "folded normalisation / K split planned for a conv the small-M kernel cannot run");
  const long long z = a.zsplit ? a.n_groups : 1;
  auto ctas = [&](int TM, int TN) { return (long long)a.B * ((a.T_y + TM - 1) / TM) * ((a.N + TN - 1) / TN) * z; };
  if (ctas(64, 64) >= 2LL * sm_count) { launch_conv_cfg<4, 16, 16>(a, st); return; }
  if (ctas(32, 32) >= 2LL * sm_count) { launch_conv_cfg<2, 8, 16>(a, st); return; }
  launch_conv_cfg<1, 8, 16>(a, st);
}

void launch_conv(avc_handle* h, const ConvArgs& a, cudaStream_t st) {
  launch_conv_simt(a, h->sm_count, st, h->conv_impl != 3);
}

// tensor-core route: decided when the plan is built (the dgrad side buffer comes from the plan's arena)
bool want_tc(const avc_handle* h, const ConvArgs& a, const TcOp& op) {
  const int impl = h->conv_impl;
  if (impl == 1 || impl == 3) return false;
  if (!tc_supported(a, op)) return false;
  if (impl == 2 || impl == 4 || impl == 5 || impl == 6 || impl == 7) return true;
  return (long long)a.B * (a.T_y + op.kmax - 1) >= h->tc_min_rows;
}

// which tcgen05 kernel: the role-swapped N = 256 kernel (conv_tc2.cuh) whenever the N = 128 kernel would need more than one
// wave of 128-row tiles; below that a 256-row tile only halves the SMs in use.  tc2: 0 auto, 1 never, 2 always (impl 6)
bool use_tc2(const TcArgs& t, int sm_count, int tc2) {
  static const int env = getenv("AVC_TC2") ? atoi(getenv("AVC_TC2")) : 0;
  const int mode = tc2 ? tc2 : env;
  if (mode == 1) return false;
  if (mode == 2) return true;
  // measured per launch at emb 128 / 512 x 80x512 (profiles/r02b_*): the N = 256 kernel wins where its 128-clk MMAs and
  // register epilogue count -- multi-tap convs with more than one wave of 128-row tiles; the N = 128 kernel keeps 1-tap convs
  // (window-loader bound either way, and its smaller tile balances better), N = 80 outputs (M is padded to 128 after the
  // swap) and dgrads whose epilogue reads an act' mask (two operand streams per tile against one accumulator hand-off)
  if (((t.Mv + kTcM - 1) / kTcM) * t.n_pass <= sm_count) return false;
  int kmax = 1;
  for (int q = 0; q < t.n_pass; ++q) {
    if (t.pass[q].N != kTcNMax) return false;
    for (int g = t.pass[q].g_begin; g < t.pass[q].g_end; ++g) kmax = std::max(kmax, t.g[g].n_taps);
  }
  if (kmax < 2) return false;
  if (t.bwd && t.Om) return false;
  return true;
}

// t.lens_y set: a ragged batch, run by the VL = true instantiations (never the CTA-pair kernel)
void launch_conv_tc(const TcArgs& t, int sm_count, cudaStream_t st, int tc2 = 0) {
  const bool vl = t.lens_y != nullptr;
  if (use_tc2(t, sm_count, tc2)) {
    const long long work = ((t.Mv + kT2N - 1) / kT2N) * t.n_pass;
    dim3 grid((unsigned)std::min<long long>(work, sm_count), 1, 1);   // persistent: one CTA per SM
    launch_k(vl ? conv_tc2_kernel<true> : conv_tc2_kernel<false>, grid, kT2Threads, tc2_smem_bytes(), st, t);
    return;
  }
  const size_t smem = tc_smem_bytes();
  const long long n_mt = (t.Mv + kTcM - 1) / kTcM;
  static const int pair_env = getenv("AVC_TC_PAIR") ? atoi(getenv("AVC_TC_PAIR")) : 0;
  if (pair_env && n_mt >= 2 && !vl) {   // CTA pairs: two M tiles of one pass per cluster, persistent over (tile pair, pass) items
    const long long work = ((n_mt + 1) / 2) * t.n_pass;
    dim3 grid(2u * (unsigned)std::min<long long>(work, sm_count / 2), 1, 1);
    launch_k_cluster(2, conv_tc_kernel_t<true>, grid, kTcThreads, smem, st, t);
    return;
  }
  const long long work = n_mt * t.n_pass;
  dim3 grid((unsigned)std::min<long long>(work, sm_count), 1, 1);   // persistent: one CTA per SM
  launch_k(vl ? conv_tc_kernel_t<false, true> : conv_tc_kernel_t<false>, grid, kTcThreads, smem, st, t);
}

void launch_tc_fold(const TcArgs& t, int sm_count, cudaStream_t st) {
  const long long n = (long long)t.B * (t.halo_l + t.halo_r) * (t.side_n / 4);
  const unsigned g = (unsigned)std::max(1LL, std::min((n + 255) / 256, (long long)sm_count * 4));
  launch_k(t.lens_y ? tc_fold_kernel<true> : tc_fold_kernel<false>, g, 256, 0, st, t.Y, t.y_bs, t.y_rs, (const float*)t.side, t.Om, t.om_bs,
           t.om_rs, t.slope, t.B, t.T_y, t.side_n, t.halo_l, t.halo_r, t.lens_y);
}

// fill the channel groups of a plain Conv1d (forward) -- K split into <=128-channel groups
void conv_groups_fwd(ConvArgs& a, const ConvW& w) {
  const int ng = (w.c_in + 127) / 128;
  if (ng > kMaxGroups) fail(AVC_ERR_INVALID, "conv c_in=%d too large", w.c_in);
  a.n_groups = ng;
  for (int g = 0; g < ng; ++g) {
    TapGroup& G = a.g[g];
    G.a_ch_off = g * 128;
    G.kc = std::min(128, w.c_in - g * 128);
    G.n_taps = w.k;
    G.off0 = -w.pl();
    G.pl = w.pl(); G.pr = w.pr();
    G.wts = w.c_in;
    G.W = w.fwd + (size_t)g * 128 * w.c_out;
  }
  a.bwd = 0; a.s = w.stride; a.N = w.c_out; a.bias = w.bias;
}

void conv_groups_bwd(ConvArgs& a, const ConvW& w) {
  const int ng = (w.c_out + 127) / 128;
  if (ng > kMaxGroups) fail(AVC_ERR_INVALID, "conv c_out=%d too large", w.c_out);
  a.n_groups = ng;
  for (int g = 0; g < ng; ++g) {
    TapGroup& G = a.g[g];
    G.a_ch_off = g * 128;
    G.kc = std::min(128, w.c_out - g * 128);
    G.n_taps = w.k;
    G.off0 = w.pl() - (w.k - 1);
    G.pl = w.pl(); G.pr = w.pr();
    G.wts = w.c_out;
    G.W = w.bwd + (size_t)g * 128 * w.c_in;
  }
  a.bwd = 1; a.s = w.stride; a.N = w.c_in; a.bias = nullptr;
}

struct Tens {   // time-major activation view
  float* p = nullptr; long long bs = 0; int rs = 0; int T = 0;
};
Tens tens(float* p, int T, int C) { return Tens{p, (long long)T * C, C, T}; }

ResArgs no_res() { ResArgs r{}; r.mode = RES_NONE; r.rf = 1; return r; }
ResArgs mk_res(const Tens& t, int mode, int rf) { ResArgs r{}; r.R = t.p; r.bs = t.bs; r.rs = t.rs; r.T_r = t.T; r.mode = mode; r.rf = rf; return r; }

int cdiv(int a, int b) { return (a + b - 1) / b; }

// =================================================================================================
// emitters: append launches to a vector
// =================================================================================================
// per-utterance lengths of a conv in a ragged batch (device int32 [B]): its input, its output and its skip tensor
struct TcLens { const int* a = nullptr; const int* y = nullptr; const int* r = nullptr; };

struct Emitter {
  avc_handle* h;
  std::vector<Launch>* out;
  Arena* mem;   // scratch that must outlive the launches (dgrad side buffers of the tensor-core path)
  // vl.y set: a conv of a ragged batch, which only the tensor-core kernels run
  void conv(const ConvArgs& a, const ConvW* cw = nullptr, const TcOp* multi = nullptr, TcLens vl = {}) {
    avc_handle* hh = h;
    ConvArgs ac = a;
    double macs = 0;
    const int g_n = ac.n_groups;
    for (int g = 0; g < g_n; ++g) macs += (double)ac.g[g].kc * ac.g[g].n_taps;
    macs *= (double)ac.B * ac.T_y * ac.N / (ac.bwd ? ac.s : 1);
    const double bytes = 4.0 * ac.B * ((double)ac.T_a * ac.g[0].kc * (ac.zsplit ? 1 : g_n) + (double)ac.T_y * ac.N * (ac.zsplit ? g_n : 1));
    Launch l;
    l.kind = LK_CONV; l.flops = 2.0 * macs; l.bytes = bytes;
    TcOp op = multi ? *multi : (cw ? tc_op_conv(*cw, ac.bwd != 0) : TcOp{});
    if (vl.y && !tc_supported(ac, op)) fail(AVC_ERR_INVALID, "ragged attacks run on the tensor-core kernels, which do not support this speaker-encoder conv");
    if (vl.y || want_tc(hh, ac, op)) {
      const size_t side_n = tc_side_floats(ac);
      float* side = side_n ? mem->f(side_n) : nullptr;
      TcArgs t = tc_make_args(ac, op, side, hh->conv_impl == 4 ? 1 : hh->conv_impl == 5 ? 4 : 3);
      t.lens_a = vl.a; t.lens_y = vl.y; t.lens_r = vl.r;
      const int smc0 = hh->sm_count;
      const int tc2 = hh->conv_impl == 6 ? 2 : hh->conv_impl == 7 ? 1 : 0;      // 6: N = 256 kernel everywhere, 7: N = 128 kernel everywhere
      l.fn = [t, smc0, tc2](cudaStream_t st) { launch_conv_tc(t, smc0, st, tc2); };
      out->push_back(std::move(l));
      if (t.side) {
        const int smc = hh->sm_count;
        Launch f;
        f.kind = LK_CONV; f.flops = 0; f.bytes = 0;
        f.fn = [t, smc](cudaStream_t st) { launch_tc_fold(t, smc, st); };
        out->push_back(std::move(f));
      }
      return;
    }
    l.fn = [hh, ac](cudaStream_t st) { launch_conv(hh, ac, st); };
    out->push_back(std::move(l));
  }
  // tile height if this conv runs on the small-M CUDA-core kernel (the only one that folds normalisations), else 0
  int small_tm_of(const ConvArgs& a, const ConvW* cw) const {
    if (h->conv_impl != 0 && h->conv_impl != 1) return 0;
    if (cw && want_tc(h, a, tc_op_conv(*cw, a.bwd != 0))) return 0;
    return small_tm(a, h->sm_count, true);
  }
  void push(int kind, double flops, double bytes, std::function<void(cudaStream_t)> fn) {
    Launch l;
    l.fn = std::move(fn); l.kind = kind; l.flops = flops; l.bytes = bytes;
    out->push_back(std::move(l));
  }
};

unsigned ew_grid(long long n4, int sm) {
  long long g = (n4 + 255) / 256;
  long long cap = (long long)sm * 8;
  return (unsigned)std::max(1LL, std::min(g, cap));
}

// forward conv through pad_layer (models.py:10-30)
ConvArgs fwd_conv_args(const ConvW& w, const Tens& in, const Tens& outT, int B, bool act, float slope) {
  ConvArgs a{};
  a.A = in.p; a.a_bs = in.bs; a.a_rs = in.rs; a.T_a = in.T;
  a.slope = slope; a.T_y = outT.T; a.B = B;
  a.Y = outT.p; a.y_bs = outT.bs; a.y_rs = outT.rs;
  a.act = act ? 1 : 0;
  a.res = no_res();
  conv_groups_fwd(a, w);
  return a;
}
// gradient w.r.t. the conv input: dy (rows of the forward output) -> dx (rows of the forward input)
ConvArgs bwd_conv_args(const ConvW& w, const Tens& dy, const Tens& dx, int B, float slope) {
  ConvArgs a{};
  a.A = dy.p; a.a_bs = dy.bs; a.a_rs = dy.rs; a.T_a = dy.T;
  a.slope = slope; a.T_y = dx.T; a.B = B;
  a.Y = dx.p; a.y_bs = dx.bs; a.y_rs = dx.rs;
  a.res = no_res();
  conv_groups_bwd(a, w);
  return a;
}

// float4 channel lanes per CTA of the norm kernels.  Measured at 2048 x 256 x 128 (profiles/README.md, round 2): strips of
// 128 B / 256 B / 512 B per row reach 66 % / 61 % / 48 % of the HBM peak forward and 66 % / 37 % / 49 % backward -- the wider
// strip streams DRAM pages better but its larger staged slice leaves fewer CTAs (loads in flight) per SM, which is what the
// kernel is bound by.  So: 128-byte strips, the wider instantiations stay for A/B runs (AVC_NORM_CL=16|32).
int norm_lanes(int sm_count, int B, int T, int C, int planes) {
  (void)sm_count; (void)B; (void)T; (void)planes;
  static const int force = getenv("AVC_NORM_CL") ? atoi(getenv("AVC_NORM_CL")) : 0;
  if ((force == 16 || force == 32) && C % (4 * force) == 0) return force;
  return 8;
}

void emit_norm_fwd(Emitter& E, const float* y, int B, int T, int C, const float* cond, int cond_bs,
                   const float* stats_in, float* stats_out, float* outp, ResArgs res, float slope) {
  NormArgs n{};
  n.y = y; n.T = T; n.C = C; n.cond = cond; n.cond_bs = cond_bs; n.stats_in = stats_in; n.stats_out = stats_out;
  n.out = outp; n.res = res; n.slope = slope;
  if (C % kNormCh) fail(AVC_ERR_INVALID, "InstanceNorm channels %d not a multiple of %d", C, kNormCh);
  const int cl = norm_lanes(E.h->sm_count, B, T, C, 1);
  dim3 grid(C / (4 * cl), B);      // channel strips fastest: the CTAs that share a row run together (same DRAM page)
  const size_t smem = (size_t)T * 4 * cl * sizeof(float);
  n.stage = smem <= (size_t)kNormSmemMax ? 1 : 0;
  const size_t dyn = n.stage ? smem : 0;
  E.push(LK_NORM, 0, 4.0 * B * T * C * ((outp ? 2 : 1) + (res.mode != RES_NONE ? 1.0 / res.rf : 0)), [n, grid, dyn, cl](cudaStream_t st) {
    if (cl == 32) launch_k(norm_act_fwd_kernel<32>, grid, 256, dyn, st, n);
    else if (cl == 16) launch_k(norm_act_fwd_kernel<16>, grid, 256, dyn, st, n);
    else launch_k(norm_act_fwd_kernel<8>, grid, 256, dyn, st, n);
  });
}

void emit_norm_bwd(Emitter& E, const float* g, const float* y, const float* stats, const float* cond, int cond_bs,
                   float* gy, float* gcond, int gcond_bs, int B, int T, int C, float slope) {
  NormBwdArgs n{};
  n.g = g; n.y = y; n.stats = stats; n.cond = cond; n.cond_bs = cond_bs; n.gy = gy; n.gcond = gcond; n.gcond_bs = gcond_bs;
  n.T = T; n.C = C; n.slope = slope;
  if (C % kNormCh) fail(AVC_ERR_INVALID, "InstanceNorm channels %d not a multiple of %d", C, kNormCh);
  const int cl = norm_lanes(E.h->sm_count, B, T, C, 2);
  dim3 grid(C / (4 * cl), B);
  const size_t smem = (size_t)T * 4 * cl * sizeof(float) * 2;
  n.stage = (gy && smem <= (size_t)kNormSmemMax) ? 1 : 0;
  const size_t dyn = n.stage ? smem : 0;
  E.push(LK_NORM, 0, 4.0 * B * T * C * (gy ? 3 : 2), [n, grid, dyn, cl](cudaStream_t st) {
    if (cl == 32) launch_k(norm_act_bwd_kernel<32>, grid, 256, dyn, st, n);
    else if (cl == 16) launch_k(norm_act_bwd_kernel<16>, grid, 256, dyn, st, n);
    else launch_k(norm_act_bwd_kernel<8>, grid, 256, dyn, st, n);
  });
}

// ---- encoder (speaker / content) ------------------------------------------------------------------
struct EncActs {
  int B = 0, T = 0;
  int Tl[AVC_MAX_BLOCKS + 1]{};
  float* cat = nullptr;            // [B,T,c_cat]; the encoder INPUT lives at cat + n_bank*c_bank (concat "x last")
  float* h0 = nullptr;
  float *h1[AVC_MAX_BLOCKS]{}, *h2[AVC_MAX_BLOCKS]{}, *hout[AVC_MAX_BLOCKS]{};
  float *tmp = nullptr, *tmp2 = nullptr;   // content encoder: raw conv outputs before InstanceNorm
  float *tail_acts = nullptr, *emb = nullptr, *gpool = nullptr;
  // backward scratch
  float *gA = nullptr, *gB = nullptr, *gH = nullptr, *gcat = nullptr, *gin = nullptr;
  // ragged batch (speaker encoder only): lens[l][b] = valid rows of utterance b at level l (device), Tl[l] their maximum.
  // Null for equal lengths.
  const int* lens[AVC_MAX_BLOCKS + 1]{};
  TcLens vl(int la, int ly, int lr = -1) const { return lens[0] ? TcLens{lens[la], lens[ly], lr >= 0 ? lens[lr] : nullptr} : TcLens{}; }
  Tens input(const EncoderW& W) const {
    return Tens{cat + W.n_bank * W.d.c_bank, (long long)T * W.c_cat, W.c_cat, T};
  }
};

// reflect padding needs pad < length for every conv INPUT (PyTorch raises otherwise, models.py:23-28): the bank sees T,
// both convs of block l see Tl[l]; the length after the last sub-sampling only feeds the pooling
bool too_short_for_encoder(const EncoderW& W, int T) {
  bool too_short = T <= W.d.bank_size / 2;
  for (int l = 0, t = T; l < W.d.n_conv_blocks; t = cdiv(t, W.d.subsample[l]), ++l) too_short = too_short || t <= W.d.kernel_size / 2;
  return too_short;
}

EncActs alloc_encoder(Arena& m, const EncoderW& W, int B, int T, bool need_bwd, bool content) {
  EncActs A;
  A.B = B; A.T = T;
  const int ch = W.d.c_h;
  A.Tl[0] = T;
  for (int l = 0; l < W.d.n_conv_blocks; ++l) A.Tl[l + 1] = cdiv(A.Tl[l], W.d.subsample[l]);
  if (too_short_for_encoder(W, T)) fail(AVC_ERR_INVALID, "utterance of %d frames is too short for reflect padding", T);
  A.cat = m.f((size_t)B * T * W.c_cat);
  A.h0 = m.f((size_t)B * T * ch);
  for (int l = 0; l < W.d.n_conv_blocks; ++l) {
    A.h1[l] = m.f((size_t)B * A.Tl[l] * ch);
    if (!content) A.h2[l] = m.f((size_t)B * A.Tl[l + 1] * ch);
    A.hout[l] = m.f((size_t)B * A.Tl[l + 1] * ch);
  }
  if (content) {
    A.tmp = m.f((size_t)B * T * ch);
    A.tmp2 = m.f((size_t)B * T * ch);
  } else {
    A.tail_acts = m.f((size_t)B * (3 * W.d.n_dense_blocks + 1) * 128);
    A.emb = m.f((size_t)B * 128);
    A.gpool = m.f((size_t)B * 128);
  }
  if (need_bwd) {
    A.gA = m.f((size_t)B * T * ch);
    A.gB = m.f((size_t)B * T * ch);
    A.gH = m.f((size_t)B * T * ch);
    A.gcat = m.f((size_t)B * T * W.c_cat);
    A.gin = m.f((size_t)B * T * W.d.c_in);
  }
  return A;
}

void emit_bank_and_inconv(Emitter& E, const EncoderW& W, const EncActs& A, bool content) {
  const float slope = W.d.neg_slope;
  const Tens x = A.input(W);
  {   // conv bank: 8 convs + act, written into their channel slots of `cat` (models.py:82-104)
    ConvArgs a{};
    a.A = x.p; a.a_bs = x.bs; a.a_rs = x.rs; a.T_a = A.T;
    a.slope = slope; a.bwd = 0; a.s = 1; a.T_y = A.T; a.B = A.B;
    a.Y = A.cat; a.y_bs = x.bs; a.y_rs = W.c_cat; a.N = W.d.c_bank; a.bias = W.bank_bias; a.act = 1;
    a.res = no_res(); a.zsplit = 1; a.n_groups = W.n_bank;
    TcOp op;
    bool tc_ok = true;
    for (int z = 0; z < W.n_bank; ++z) {
      const ConvW& w = W.bank[z];
      a.g[z] = TapGroup{w.fwd, 0, w.c_in, w.k, -w.pl(), w.pl(), w.pr(), w.c_in};
      const TcPack& pk = w.tc_fwd[0];
      const int gi = (pk.ok && pk.n_chunks == 1) ? op.add_group(pk.blocks[0], 0, w.c_in, w.k, 1, -w.pl()) : -1;
      tc_ok = tc_ok && gi >= 0 && op.add_pass(gi, gi + 1, pk.cn[0], z * W.d.c_bank, 1, 0);   // one pass per bank conv
    }
    if (!tc_ok) op = TcOp{};
    E.conv(a, nullptr, &op, A.vl(0, 0));
  }
  {   // 1x1 in-conv over the concatenation (models.py:192 / :337)
    Tens cat{A.cat, x.bs, W.c_cat, A.T};
    Tens outT = tens(content ? A.tmp : A.h0, A.T, W.d.c_h);
    ConvArgs a = fwd_conv_args(W.in_conv, cat, outT, A.B, !content, slope);
    E.conv(a, &W.in_conv, nullptr, A.vl(0, 0));
    if (content) emit_norm_fwd(E, A.tmp, A.B, A.T, W.d.c_h, nullptr, 0, nullptr, nullptr, A.h0, no_res(), slope);
  }
}

void emit_encoder_blocks_fwd(Emitter& E, const EncoderW& W, const EncActs& A, bool content) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h;
  const float* hin = A.h0;
  for (int l = 0; l < W.d.n_conv_blocks; ++l) {
    const int Ti = A.Tl[l], To = A.Tl[l + 1], sub = W.d.subsample[l];
    Tens in = tens(const_cast<float*>(hin), Ti, ch);
    ResArgs res = mk_res(in, sub > 1 ? RES_POOL : RES_SAME, sub);
    if (!content) {
      ConvArgs a1 = fwd_conv_args(W.c1[l], in, tens(A.h1[l], Ti, ch), A.B, true, slope);
      E.conv(a1, &W.c1[l], nullptr, A.vl(l, l));
      ConvArgs a2 = fwd_conv_args(W.c2[l], tens(A.h1[l], Ti, ch), tens(A.hout[l], To, ch), A.B, true, slope);
      a2.Y2 = A.h2[l]; a2.y2_bs = (long long)To * ch; a2.y2_rs = ch;
      a2.res = res;
      E.conv(a2, &W.c2[l], nullptr, A.vl(l, l + 1, l));
    } else {
      ConvArgs a1 = fwd_conv_args(W.c1[l], in, tens(A.tmp, Ti, ch), A.B, false, slope);
      E.conv(a1, &W.c1[l]);
      emit_norm_fwd(E, A.tmp, A.B, Ti, ch, nullptr, 0, nullptr, nullptr, A.h1[l], no_res(), slope);
      ConvArgs a2 = fwd_conv_args(W.c2[l], tens(A.h1[l], Ti, ch), tens(A.tmp2, To, ch), A.B, false, slope);
      E.conv(a2, &W.c2[l]);
      emit_norm_fwd(E, A.tmp2, A.B, To, ch, nullptr, 0, nullptr, nullptr, A.hout[l], res, slope);
    }
    hin = A.hout[l];
  }
}

TailArgs tail_args(const EncoderW& W, const EncActs& A) {
  TailArgs t{};
  const int nb = W.d.n_conv_blocks;
  t.h = nb ? A.hout[nb - 1] : A.h0;
  t.T_h = A.Tl[nb]; t.h_rs = W.d.c_h; t.h_bs = (long long)t.T_h * W.d.c_h;
  t.n_dense = W.d.n_dense_blocks;
  for (int l = 0; l < t.n_dense; ++l) {
    t.Wt1[l] = W.Wt1[l]; t.Wt2[l] = W.Wt2[l]; t.W1[l] = W.W1[l]; t.W2[l] = W.W2[l]; t.b1[l] = W.b1[l]; t.b2[l] = W.b2[l];
  }
  t.Wto = W.Wto; t.Wo = W.Wo; t.bo = W.bo;
  t.slope = W.d.neg_slope;
  t.acts = A.tail_acts; t.emb = A.emb; t.gpool = A.gpool;
  t.lens_h = A.lens[nb];
  return t;
}

void emit_tail(Emitter& E, const TailArgs& t, int B) {
  // small batches: a cluster of 8 CTAs per utterance with the matrix slices resident (se_tail_cluster_kernel)
  const int n_mats = (2 * t.n_dense + 1) * (((t.mode & TAIL_FWD) ? 1 : 0) + ((t.mode & TAIL_BWD) ? 1 : 0));
  const size_t csm = (size_t)n_mats * kTclMatBytes;
  static const bool no_cluster = getenv("AVC_NO_TAIL_CLUSTER") != nullptr;
  const bool cluster = !no_cluster && B * kTclN <= E.h->sm_count && csm + 4096 <= kSmemMax;
  const bool vl = t.lens_h != nullptr;
  E.push(LK_TAIL, 2.0 * B * 128 * 128 * (2 * t.n_dense + 1) * (((t.mode & TAIL_FWD) ? 1 : 0) + ((t.mode & TAIL_BWD) ? 1 : 0)), 0, [t, B, cluster, csm, vl](cudaStream_t st) {
    if (cluster) launch_k_cluster(kTclN, vl ? se_tail_cluster_kernel<true> : se_tail_cluster_kernel<false>, B * kTclN, 128, csm, st, t);
    else launch_k(vl ? se_tail_kernel<true> : se_tail_kernel<false>, B, 1024, kTailSmem, st, t);
  });
}

// speaker-encoder backward from gpool ([B,128], gradient of every pooled row) down to d input
// partial input gradients of a K-split conv-bank dgrad (small-M plans): the consumer adds p[0..n) to gin, in order
struct GradParts { const float* p[kMaxZk - 1] = {nullptr, nullptr}; int n = 0; };

// `parts` non-null: the caller's consumer of gin can add partials, so the bank dgrad may split its K over blockIdx.z
void emit_speaker_bwd(Emitter& E, const EncoderW& W, const EncActs& A, const Tens& gin, GradParts* parts = nullptr) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h, nb = W.d.n_conv_blocks;
  Tens gout{A.gpool, (long long)ch, 0, A.Tl[nb]};   // broadcast over time (row stride 0)
  float* pingpong[2] = {A.gA, A.gB};
  for (int l = nb - 1; l >= 0; --l) {
    const int Ti = A.Tl[l], To = A.Tl[l + 1], sub = W.d.subsample[l];
    gout.T = To;
    // through act + second conv: gH = (conv2^T (gout * act'(h2))) * act'(h1)
    Tens gH = tens(A.gH, Ti, ch);
    ConvArgs a2 = bwd_conv_args(W.c2[l], gout, gH, A.B, slope);
    a2.Mk = A.h2[l]; a2.m_bs = (long long)To * ch; a2.m_rs = ch;
    a2.Om = A.h1[l]; a2.om_bs = (long long)Ti * ch; a2.om_rs = ch;
    E.conv(a2, &W.c2[l], nullptr, A.vl(l + 1, l));
    // through the first conv, plus the skip path (avg-pool backward when sub-sampled)
    Tens gx = tens(pingpong[l & 1], Ti, ch);
    ConvArgs a1 = bwd_conv_args(W.c1[l], gH, gx, A.B, slope);
    a1.res = mk_res(gout, sub > 1 ? RES_POOL_BWD : RES_SAME, sub);
    E.conv(a1, &W.c1[l], nullptr, A.vl(l, l, l + 1));
    gout = gx;
  }
  if (nb == 0) fail(AVC_ERR_INVALID, "n_conv_blocks must be > 0");
  {   // 1x1 in-conv: gcat = (gout * act'(h0)) W_in
    Tens gcat = tens(A.gcat, A.T, W.c_cat);
    ConvArgs a = bwd_conv_args(W.in_conv, gout, gcat, A.B, slope);
    a.Mk = A.h0; a.m_bs = (long long)A.T * ch; a.m_rs = ch;
    // Batched plans: a [B*T, 128] x [128, 1104] GEMM whose nine 128-column passes re-gathered the same A window in
    // conv_tc_kernel (12 % tensor pipe, the loaders starve a 1-tap pass).  Here the masked gradient is split into hi / lo
    // planes by one elementwise pass and conv2d_tc_kernel streams both operands with TMA tensor loads (3xTF32).
    static const bool no_tma = getenv("AVC_NO_TMA_INCONV") != nullptr;
    const bool contiguous = gout.rs == ch && gout.bs == (long long)A.T * ch;
    // (ragged batches too: a 1x1 GEMM over the padded rows, whose dead rows only reach dead rows of gcat)
    if (!no_tma && W.in_conv.fwd_h && contiguous && ch % 32 == 0 && (A.lens[0] || want_tc(E.h, a, tc_op_conv(W.in_conv, true)))) {
      const size_t n = (size_t)A.B * A.T * ch;
      float* ph = E.mem->f(n); float* pl = E.mem->f(n);
      const float* g = gout.p; const float* mk = A.h0;
      const unsigned sg = ew_grid((long long)n / 4, E.h->sm_count);
      E.push(LK_CONV, 0, 16.0 * n, [=](cudaStream_t st) {
        wt_split_mask_kernel<<<sg, 256, 0, st>>>(g, mk, slope, ph, pl, (long long)n / 4);
        CK(cudaGetLastError());
      });
      C2Args c{};
      c.B = A.B; c.Hb = 1; c.Wb = A.T; c.a_wmul = c.a_hmul = 1; c.n_taps = 1;
      c.Ci = ch; c.Cop = W.c_cat; c.y = gcat.p; c.Ho = 1; c.Wo = A.T; c.Co = W.c_cat;
      c.oh_mul = c.ow_mul = 1; c.ksplit = 1;
      c2_pick_boxes(c);
      const WtOperand X{ph, pl, ch, A.T, 1, A.B, 1, 1};
      const float* wh = W.in_conv.fwd_h; const float* wl = W.in_conv.fwd_l;
      const int rows = W.c_cat, smc = E.h->sm_count;
      E.push(LK_CONV, 2.0 * A.B * A.T * ch * W.c_cat, 4.0 * A.B * A.T * (ch + W.c_cat), [=](cudaStream_t st) {
        launch_conv2d_tc(X, wh, wl, ch, rows, c, smc, st, 1);
      });
    } else {
      E.conv(a, &W.in_conv, nullptr, A.vl(0, 0));
    }
  }
  {   // conv bank: sum of the 8 transposed convs of (gcat_k * act'(cat_k)) + pass-through slice
    ConvArgs a{};
    a.A = A.gcat; a.a_bs = (long long)A.T * W.c_cat; a.a_rs = W.c_cat; a.T_a = A.T;
    a.Mk = A.cat; a.m_bs = a.a_bs; a.m_rs = W.c_cat;
    a.slope = slope; a.bwd = 1; a.s = 1; a.T_y = A.T; a.B = A.B;
    a.Y = gin.p; a.y_bs = gin.bs; a.y_rs = gin.rs; a.N = W.d.c_in;
    Tens pass{A.gcat + W.n_bank * W.d.c_bank, a.a_bs, W.c_cat, A.T};
    a.res = mk_res(pass, RES_SAME, 1);
    a.n_groups = W.n_bank;
    TcOp op;
    bool tc_ok = true;
    int PL = 0;
    for (int z = 0; z < W.n_bank; ++z) PL = std::max(PL, W.bank[z].pl());
    for (int z = 0; z < W.n_bank; ++z) {
      const ConvW& w = W.bank[z];
      a.g[z] = TapGroup{w.bwd, z * W.d.c_bank, w.c_out, w.k, w.pl() - (w.k - 1), w.pl(), w.pr(), w.c_out};
      const TcPack& pk = w.tc_bwd[0];
      tc_ok = tc_ok && pk.ok && pk.n_chunks == 1 &&
              op.add_group(pk.blocks[0], z * W.d.c_bank, w.c_out, w.k, 1, w.pl() - (w.k - 1) - PL) >= 0;
    }
    tc_ok = tc_ok && op.add_pass(0, op.n_groups, W.bank[0].tc_bwd[0].cn[0], 0, 1, -PL);   // one pass sums the 8 transposed convs
    if (!tc_ok) op = TcOp{};
    static const bool no_zk = getenv("AVC_NO_KSPLIT") != nullptr;
    if (parts && !no_zk && !A.lens[0] && W.n_bank >= kMaxZk && !want_tc(E.h, a, op) && E.small_tm_of(a, nullptr)) {
      // batch-1 plans: this conv contracts K = sum_k k*c_bank (36 weight slabs for the 8-kernel bank), four times the longest
      // other layer, on too few CTAs.  Split K into kMaxZk balanced ranges of whole groups (longest-processing-time first).
      ConvArgs sp = a;
      int order[kMaxGroups], bin_of[kMaxGroups], load[kMaxZk] = {0};
      for (int z = 0; z < W.n_bank; ++z) order[z] = z;
      std::sort(order, order + W.n_bank, [&](int x, int y) { return a.g[x].n_taps > a.g[y].n_taps; });
      for (int i = 0; i < W.n_bank; ++i) {
        int best = 0;
        for (int q = 1; q < kMaxZk; ++q) if (load[q] < load[best]) best = q;
        bin_of[order[i]] = best; load[best] += a.g[order[i]].n_taps;
      }
      int n = 0;
      for (int q = 0; q < kMaxZk; ++q) {
        sp.zk_lo[q] = n;
        for (int i = 0; i < W.n_bank; ++i) if (bin_of[order[i]] == q) sp.g[n++] = a.g[order[i]];
        sp.zk_hi[q] = n;
      }
      sp.zk = kMaxZk;
      if (E.small_tm_of(sp, nullptr)) {
        for (int q = 0; q + 1 < kMaxZk; ++q) {
          sp.y_part[q] = E.mem->f((size_t)A.B * A.T * W.d.c_in);
          parts->p[q] = sp.y_part[q];
        }
        parts->n = kMaxZk - 1;
        E.conv(sp, nullptr, nullptr);
        return;
      }
    }
    E.conv(a, nullptr, &op, A.vl(0, 0, 0));
  }
}

// ---- decoder ------------------------------------------------------------------------------------------
struct DecActs {
  int B = 0, L = 0, nb = 0;
  int Td[AVC_MAX_BLOCKS + 1]{};
  float* z = nullptr;                 // content code mu [B,L,c_in]
  float* c0 = nullptr;                // in-conv raw output
  float* h[AVC_MAX_BLOCKS + 1]{};     // block inputs/outputs
  float *c1[AVC_MAX_BLOCKS]{}, *c2[AVC_MAX_BLOCKS]{}, *r1[AVC_MAX_BLOCKS]{};
  float *st1[AVC_MAX_BLOCKS]{}, *st2[AVC_MAX_BLOCKS]{};
  float *cond = nullptr, *gcond = nullptr, *gemb_parts = nullptr;
  float *gh[2]{}, *gy = nullptr, *gr1 = nullptr;
  int T_out() const { return Td[nb]; }
};

DecActs alloc_decoder(Arena& m, const DecoderW& W, int B, int L, bool need_bwd) {
  DecActs A;
  A.B = B; A.L = L; A.nb = W.d.n_conv_blocks;
  const int ch = W.d.c_h;
  if (L <= W.d.kernel_size / 2) fail(AVC_ERR_INVALID, "content code of %d frames is too short for reflect padding", L);
  A.Td[0] = L;
  for (int l = 0; l < A.nb; ++l) A.Td[l + 1] = A.Td[l] * W.d.upsample[l];
  A.z = m.f((size_t)B * L * W.d.c_in);
  A.c0 = m.f((size_t)B * L * ch);
  A.h[0] = m.f((size_t)B * L * ch);
  for (int l = 0; l < A.nb; ++l) {
    A.c1[l] = m.f((size_t)B * A.Td[l] * ch);
    A.r1[l] = m.f((size_t)B * A.Td[l] * ch);
    A.c2[l] = m.f((size_t)B * A.Td[l + 1] * ch);
    A.h[l + 1] = m.f((size_t)B * A.Td[l + 1] * ch);
    A.st1[l] = m.f((size_t)B * ch * 2);
    A.st2[l] = m.f((size_t)B * ch * 2);
  }
  A.cond = m.f((size_t)B * 2 * A.nb * 2 * ch);
  if (need_bwd) {
    A.gcond = m.f((size_t)B * 2 * A.nb * 2 * ch);
    A.gemb_parts = m.f((size_t)B * 2 * A.nb * 128);
    const size_t big = (size_t)B * A.Td[A.nb] * ch;
    A.gh[0] = m.f(big); A.gh[1] = m.f(big); A.gy = m.f(big); A.gr1 = m.f(big);
  }
  return A;
}

// loop-invariant prefix: h0 = act(IN(in_conv(z))), c1[0] = conv1_0(h0) and its statistics (models.py:413-418)
void emit_decoder_const(Emitter& E, const DecoderW& W, const DecActs& A) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h;
  ConvArgs a = fwd_conv_args(W.in_conv, tens(A.z, A.L, W.d.c_in), tens(A.c0, A.L, ch), A.B, false, slope);
  E.conv(a, &W.in_conv);
  emit_norm_fwd(E, A.c0, A.B, A.L, ch, nullptr, 0, nullptr, nullptr, A.h[0], no_res(), slope);
  ConvArgs a1 = fwd_conv_args(W.c1[0], tens(A.h[0], A.L, ch), tens(A.c1[0], A.L, ch), A.B, false, slope);
  E.conv(a1, &W.c1[0]);
  emit_norm_fwd(E, A.c1[0], A.B, A.L, ch, nullptr, 0, nullptr, A.st1[0], nullptr, no_res(), slope);
}

AffineArgs affine_args(const DecoderW& W, const DecActs& A, const float* emb) {
  AffineArgs f{};
  f.L = 2 * A.nb;
  for (int l = 0; l < f.L; ++l) { f.Wt[l] = W.aWt[l]; f.W[l] = W.aW[l]; f.bias[l] = W.ab[l]; }
  f.emb = emb; f.cond = A.cond; f.gcond = A.gcond; f.gemb_parts = A.gemb_parts;
  return f;
}

// emb-dependent part of the decoder forward (models.py:417-434); `outT` receives the [B,T,c_out] mel
// ---- folded decoder (batch-1 plans): no separate normalisation launches --------------------------------
// A normalisation whose application is deferred into the window load of the next conv (conv_simt.cuh: FoldPro).
struct PendingNorm {
  float* y; int T;                 // raw conv output viewed [B][T][ch]
  const float* cond;               // AdaIN row of this layer
  const float* stats; float* stats_out;
  float* part; int n_part, tm, up, part_T;
  ResArgs res; float* out;
};

bool fold_enabled(const DecoderW& W) {
  static const bool off = getenv("AVC_NO_FOLD") != nullptr;
  return !off && W.d.c_h <= 128 && W.d.c_h % 32 == 0;
}

// consumer side: conv reads act(AdaIN(IN(P.y))) [+res] through its window
void fold_fwd_in(ConvArgs& a, const PendingNorm& P, int ch, int cb) {
  a.A = P.y; a.a_bs = (long long)P.T * ch; a.a_rs = ch; a.T_a = P.T;
  FoldPro& f = a.pro;
  f.mode = 1; f.C = ch; f.T = P.T; f.part = P.part; f.n_part = P.n_part; f.part_tm = P.tm; f.part_up = P.up; f.part_T = P.part_T;
  f.stats = P.stats; f.stats_out = P.stats_out; f.cond = P.cond; f.cond_bs = cb; f.res = P.res; f.out = P.out;
}
// producer side: conv also writes the per-tile partial statistics of its output
float* fold_fwd_out(Emitter& E, ConvArgs& a, int tm, int ch, int* n_part) {
  const int np = cdiv(a.T_y, tm) * (a.N / ch);
  if (np > kFoldMaxPart || a.T_y % tm) { *n_part = 0; return nullptr; }   // ragged tiles: the consumer assumes equal row counts
  float* part = E.mem->f((size_t)a.B * np * ch * 2);
  a.epi.mode = 1; a.epi.C = ch; a.epi.part = part; a.epi.n_part = np;
  *n_part = np;
  return part;
}

bool emit_decoder_fwd_folded(Emitter& E, const DecoderW& W, const DecActs& A, const float* emb, const Tens& outT) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h, L2 = 2 * A.nb, cb = L2 * 2 * ch;
  if (!fold_enabled(W)) return false;
  AffineArgs f = affine_args(W, A, emb);
  dim3 ag(A.B, L2);
  E.push(LK_AFFINE, 2.0 * A.B * L2 * 256 * 128, 0, [f, ag](cudaStream_t st) { launch_k(affine_fwd_kernel, ag, 1024, 0, st, f); });
  PendingNorm P{};
  P.y = A.c1[0]; P.T = A.Td[0]; P.cond = A.cond; P.stats = A.st1[0]; P.res = no_res();   // c1[0] and its statistics are loop constants
  for (int l = 0; l < A.nb; ++l) {
    const int Ti = A.Td[l], To = A.Td[l + 1], up = W.d.upsample[l];
    if (up != 1 && up != 2) return false;
    if (l > 0) {
      ConvArgs a1 = fwd_conv_args(W.c1[l], tens(A.h[l], Ti, ch), tens(A.c1[l], Ti, ch), A.B, false, slope);
      fold_fwd_in(a1, P, ch, cb);
      const int tm = E.small_tm_of(a1, &W.c1[l]);
      if (!tm || a1.s != 1) return false;
      PendingNorm Q{};
      Q.part = fold_fwd_out(E, a1, tm, ch, &Q.n_part);
      if (!Q.part) return false;
      Q.y = A.c1[l]; Q.T = Ti; Q.cond = A.cond + (2 * l) * 2 * ch; Q.stats_out = A.st1[l]; Q.tm = tm; Q.up = 1; Q.part_T = Ti; Q.res = no_res();
      E.conv(a1, &W.c1[l]);
      P = Q;
    }
    ConvArgs a2 = fwd_conv_args(W.c2[l], tens(A.r1[l], Ti, ch), Tens{A.c2[l], (long long)Ti * ch * up, ch * up, Ti}, A.B, false, slope);
    fold_fwd_in(a2, P, ch, cb);
    const int tm2 = E.small_tm_of(a2, &W.c2[l]);
    if (!tm2 || a2.s != 1 || a2.N != ch * up) return false;
    PendingNorm Q{};
    Q.part = fold_fwd_out(E, a2, tm2, ch, &Q.n_part);
    if (!Q.part) return false;
    Q.y = A.c2[l]; Q.T = To; Q.cond = A.cond + (2 * l + 1) * 2 * ch; Q.stats_out = A.st2[l]; Q.tm = tm2; Q.up = up; Q.part_T = Ti;
    Q.res = mk_res(tens(A.h[l], Ti, ch), up > 1 ? RES_UP : RES_SAME, up);
    Q.out = l + 1 < A.nb ? A.h[l + 1] : nullptr;      // h[l+1] is read again as the skip connection of block l+1
    E.conv(a2, &W.c2[l]);
    P = Q;
  }
  ConvArgs ao = fwd_conv_args(W.out_conv, tens(A.h[A.nb], A.Td[A.nb], ch), outT, A.B, false, slope);
  fold_fwd_in(ao, P, ch, cb);
  if (!E.small_tm_of(ao, &W.out_conv) || ao.s != 1) return false;
  E.conv(ao, &W.out_conv);
  return true;
}

void emit_decoder_fwd_plain(Emitter& E, const DecoderW& W, const DecActs& A, const float* emb, const Tens& outT);
void emit_decoder_fwd(Emitter& E, const DecoderW& W, const DecActs& A, const float* emb, const Tens& outT) {
  const size_t mark = E.out->size();
  if (emit_decoder_fwd_folded(E, W, A, emb, outT)) return;
  E.out->resize(mark);
  emit_decoder_fwd_plain(E, W, A, emb, outT);
}

void emit_decoder_fwd_plain(Emitter& E, const DecoderW& W, const DecActs& A, const float* emb, const Tens& outT) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h, L2 = 2 * A.nb, cb = L2 * 2 * ch;
  AffineArgs f = affine_args(W, A, emb);
  dim3 ag(A.B, L2);
  E.push(LK_AFFINE, 2.0 * A.B * L2 * 256 * 128, 0, [f, ag](cudaStream_t st) { launch_k(affine_fwd_kernel, ag, 1024, 0, st, f); });
  for (int l = 0; l < A.nb; ++l) {
    const int Ti = A.Td[l], To = A.Td[l + 1], up = W.d.upsample[l];
    if (l > 0) {
      ConvArgs a1 = fwd_conv_args(W.c1[l], tens(A.h[l], Ti, ch), tens(A.c1[l], Ti, ch), A.B, false, slope);
      E.conv(a1, &W.c1[l]);
    }
    emit_norm_fwd(E, A.c1[l], A.B, Ti, ch, A.cond + (2 * l) * 2 * ch, cb, l == 0 ? A.st1[0] : nullptr,
                  l == 0 ? nullptr : A.st1[l], A.r1[l], no_res(), slope);
    // second conv: c_h -> c_h*up channels; the packed weights are channel-permuted so that the
    // [Ti, ch*up] result IS the pixel-shuffled [Ti*up, ch] tensor (models.py:33-49)
    ConvArgs a2 = fwd_conv_args(W.c2[l], tens(A.r1[l], Ti, ch), Tens{A.c2[l], (long long)Ti * ch * up, ch * up, Ti}, A.B, false, slope);
    E.conv(a2, &W.c2[l]);
    ResArgs res = mk_res(tens(A.h[l], Ti, ch), up > 1 ? RES_UP : RES_SAME, up);
    emit_norm_fwd(E, A.c2[l], A.B, To, ch, A.cond + (2 * l + 1) * 2 * ch, cb, nullptr, A.st2[l], A.h[l + 1], res, slope);
  }
  ConvArgs ao = fwd_conv_args(W.out_conv, tens(A.h[A.nb], A.Td[A.nb], ch), outT, A.B, false, slope);
  E.conv(ao, &W.out_conv);
}

// decoder backward: gout = dL/d(decoder output) -> gemb_parts [B, 2*nb, 128]
// producer side (backward): the dgrad conv also writes per-tile S1/S2 of the normalisation its output flows into
bool fold_bwd_out(Emitter& E, ConvArgs& a, const ConvW* cw, const float* y, const float* stats, const float* cond, int ch, int cb,
                  float** part, int* n_part) {
  const int tm = E.small_tm_of(a, cw);
  if (!tm || a.N != ch) return false;
  const int np = cdiv(a.T_y, tm);
  if (np > kFoldMaxPart) return false;
  *part = E.mem->f((size_t)a.B * np * ch * 2);
  *n_part = np;
  a.epi.mode = 2; a.epi.C = ch; a.epi.part = *part; a.epi.n_part = np; a.epi.y = y; a.epi.stats = stats; a.epi.cond = cond; a.epi.cond_bs = cb;
  return true;
}
void fold_bwd_in(ConvArgs& a, const float* part, int n_part, int T, const float* y, const float* stats, const float* cond,
                 float* gcond, int ch, int cb) {
  FoldPro& f = a.pro;
  f.mode = 2; f.C = ch; f.T = T; f.part = part; f.n_part = n_part; f.stats = stats; f.cond = cond; f.cond_bs = cb; f.y = y;
  f.gcond = gcond; f.gcond_bs = cb; f.res = no_res();
}

bool emit_decoder_bwd_folded(Emitter& E, const DecoderW& W, const DecActs& A, const Tens& gout) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h, L2 = 2 * A.nb, cb = L2 * 2 * ch;
  if (!fold_enabled(W)) return false;
  int cur = 0;
  float* part = nullptr; int n_part = 0;
  {
    ConvArgs a = bwd_conv_args(W.out_conv, gout, tens(A.gh[cur], A.Td[A.nb], ch), A.B, slope);
    if (!fold_bwd_out(E, a, &W.out_conv, A.c2[A.nb - 1], A.st2[A.nb - 1], A.cond + (2 * (A.nb - 1) + 1) * 2 * ch, ch, cb, &part, &n_part)) return false;
    E.conv(a, &W.out_conv);
  }
  for (int l = A.nb - 1; l >= 0; --l) {
    const int Ti = A.Td[l], To = A.Td[l + 1], up = W.d.upsample[l];
    Tens gh = tens(A.gh[cur], To, ch);
    // dgrad of conv2: its window is d/d(c2[l]) of act(AdaIN(IN(c2[l]))) applied to gh, viewed [Ti, ch*up]
    ConvArgs a2 = bwd_conv_args(W.c2[l], Tens{gh.p, (long long)Ti * ch * up, ch * up, Ti}, tens(A.gr1, Ti, ch), A.B, slope);
    fold_bwd_in(a2, part, n_part, To, A.c2[l], A.st2[l], A.cond + (2 * l + 1) * 2 * ch, A.gcond + (2 * l + 1) * 2 * ch, ch, cb);
    if (a2.s != 1) return false;
    if (l > 0) {
      if (!fold_bwd_out(E, a2, &W.c2[l], A.c1[l], A.st1[l], A.cond + (2 * l) * 2 * ch, ch, cb, &part, &n_part)) return false;
    } else if (!E.small_tm_of(a2, &W.c2[l])) {
      return false;
    }
    E.conv(a2, &W.c2[l]);
    if (l > 0) {
      Tens gnext = tens(A.gh[cur ^ 1], Ti, ch);
      ConvArgs a1 = bwd_conv_args(W.c1[l], tens(A.gr1, Ti, ch), gnext, A.B, slope);
      a1.res = mk_res(gh, up > 1 ? RES_UP_BWD : RES_SAME, up);
      fold_bwd_in(a1, part, n_part, Ti, A.c1[l], A.st1[l], A.cond + (2 * l) * 2 * ch, A.gcond + (2 * l) * 2 * ch, ch, cb);
      if (a1.s != 1) return false;
      if (!fold_bwd_out(E, a1, &W.c1[l], A.c2[l - 1], A.st2[l - 1], A.cond + (2 * (l - 1) + 1) * 2 * ch, ch, cb, &part, &n_part)) return false;
      E.conv(a1, &W.c1[l]);
      cur ^= 1;
    } else {
      // first AdaIN of the decoder: c1[0] is a loop constant, only d cond is needed
      emit_norm_bwd(E, A.gr1, A.c1[0], A.st1[0], A.cond, cb, nullptr, A.gcond, cb, A.B, Ti, ch, slope);
    }
  }
  AffineArgs f = affine_args(W, A, nullptr);
  dim3 ag(A.B, L2);
  E.push(LK_AFFINE, 2.0 * A.B * L2 * 256 * 128, 0, [f, ag](cudaStream_t st) { launch_k(affine_bwd_kernel, ag, 1024, 0, st, f); });
  return true;
}

void emit_decoder_bwd_plain(Emitter& E, const DecoderW& W, const DecActs& A, const Tens& gout);
void emit_decoder_bwd(Emitter& E, const DecoderW& W, const DecActs& A, const Tens& gout) {
  const size_t mark = E.out->size();
  if (emit_decoder_bwd_folded(E, W, A, gout)) return;
  E.out->resize(mark);
  emit_decoder_bwd_plain(E, W, A, gout);
}

void emit_decoder_bwd_plain(Emitter& E, const DecoderW& W, const DecActs& A, const Tens& gout) {
  const float slope = W.d.neg_slope;
  const int ch = W.d.c_h, L2 = 2 * A.nb, cb = L2 * 2 * ch;
  int cur = 0;
  {
    ConvArgs a = bwd_conv_args(W.out_conv, gout, tens(A.gh[cur], A.Td[A.nb], ch), A.B, slope);
    E.conv(a, &W.out_conv);
  }
  for (int l = A.nb - 1; l >= 0; --l) {
    const int Ti = A.Td[l], To = A.Td[l + 1], up = W.d.upsample[l];
    Tens gh = tens(A.gh[cur], To, ch);
    emit_norm_bwd(E, gh.p, A.c2[l], A.st2[l], A.cond + (2 * l + 1) * 2 * ch, cb, A.gy, A.gcond + (2 * l + 1) * 2 * ch, cb,
                  A.B, To, ch, slope);
    ConvArgs a2 = bwd_conv_args(W.c2[l], Tens{A.gy, (long long)Ti * ch * up, ch * up, Ti}, tens(A.gr1, Ti, ch), A.B, slope);
    E.conv(a2, &W.c2[l]);
    emit_norm_bwd(E, A.gr1, A.c1[l], A.st1[l], A.cond + (2 * l) * 2 * ch, cb, l > 0 ? A.gy : nullptr,
                  A.gcond + (2 * l) * 2 * ch, cb, A.B, Ti, ch, slope);
    if (l > 0) {
      Tens gnext = tens(A.gh[cur ^ 1], Ti, ch);
      ConvArgs a1 = bwd_conv_args(W.c1[l], tens(A.gy, Ti, ch), gnext, A.B, slope);
      a1.res = mk_res(gh, up > 1 ? RES_UP_BWD : RES_SAME, up);
      E.conv(a1, &W.c1[l]);
      cur ^= 1;
    }
  }
  AffineArgs f = affine_args(W, A, nullptr);
  dim3 ag(A.B, L2);
  E.push(LK_AFFINE, 2.0 * A.B * L2 * 256 * 128, 0, [f, ag](cudaStream_t st) { launch_k(affine_bwd_kernel, ag, 1024, 0, st, f); });
}

// ---- misc launch helpers ------------------------------------------------------------------------------
void emit_layout_in(Emitter& E, const float* src, const int64_t s[3], const Tens& dst, int B, int C) {
  const long long sb = s[0], sc = s[1], st_ = s[2];
  const long long n = (long long)B * dst.T * C;
  const Tens d = dst;
  E.push(LK_LAYOUT, 0, 8.0 * n, [=](cudaStream_t st) {
    launch_k(layout_in_kernel, (unsigned)((n + 255) / 256), 256, 0, st, src, sb, sc, st_, d.p, d.bs, d.rs, B, C, d.T);
  });
}
void emit_layout_out(Emitter& E, const Tens& src, float* dst, const int64_t s[3], int B, int C) {
  const long long sb = s[0], sc = s[1], st_ = s[2];
  const long long n = (long long)B * src.T * C;
  const Tens d = src;
  E.push(LK_LAYOUT, 0, 8.0 * n, [=](cudaStream_t st) {
    launch_k(layout_out_kernel, (unsigned)((n + 255) / 256), 256, 0, st, d.p, d.bs, d.rs, dst, sb, sc, st_, B, C, d.T);
  });
}
// the same with the caller's tensor read through the plan at launch time (IoBind): cached plans are rebound, not rebuilt
void emit_layout_in_io(Emitter& E, const float* const* src, const int64_t* s, const Tens& dst, int B, int C) {
  const long long n = (long long)B * dst.T * C;
  const Tens d = dst;
  E.push(LK_LAYOUT, 0, 8.0 * n, [=](cudaStream_t st) {
    launch_k(layout_in_kernel, (unsigned)((n + 255) / 256), 256, 0, st, *src, (long long)s[0], (long long)s[1], (long long)s[2], d.p, d.bs, d.rs, B, C, d.T);
  });
}
void emit_layout_out_io(Emitter& E, const Tens& src, float* const* dst, const int64_t* s, int B, int C) {
  const long long n = (long long)B * src.T * C;
  const Tens d = src;
  E.push(LK_LAYOUT, 0, 8.0 * n, [=](cudaStream_t st) {
    if (!*dst) return;
    launch_k(layout_out_kernel, (unsigned)((n + 255) / 256), 256, 0, st, d.p, d.bs, d.rs, *dst, (long long)s[0], (long long)s[1], (long long)s[2], B, C, d.T);
  });
}
// ragged batches: the caller's packed [sum_b T_b, C] (row offsets `offs`, device [B+1]) <-> the padded slots of dst / src
void emit_layout_in_varlen_io(Emitter& E, const float* const* src, const int* offs, const Tens& dst, int B, int C, long long rows) {
  const Tens d = dst;
  const unsigned gx = (unsigned)cdiv(d.T * C, 256);
  E.push(LK_LAYOUT, 0, 8.0 * rows * C, [=](cudaStream_t st) {
    launch_k(layout_in_varlen_kernel, dim3(gx, B), 256, 0, st, *src, offs, d.p, d.bs, d.rs, C);
  });
}
void emit_layout_out_varlen_io(Emitter& E, const Tens& src, const int* offs, float* const* dst, int B, int C, long long rows) {
  const Tens d = src;
  const unsigned gx = (unsigned)cdiv(d.T * C, 256);
  E.push(LK_LAYOUT, 0, 8.0 * rows * C, [=](cudaStream_t st) {
    if (!*dst) return;
    launch_k(layout_out_varlen_kernel, dim3(gx, B), 256, 0, st, (const float*)d.p, d.bs, d.rs, offs, *dst, C);
  });
}
void emit_copy(Emitter& E, float* dst, const float* src, size_t n) {
  E.push(LK_COPY, 0, 8.0 * n, [=](cudaStream_t st) { CK(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st)); });
}
void emit_zero(Emitter& E, void* dst, size_t bytes) {
  E.push(LK_COPY, 0, (double)bytes, [=](cudaStream_t st) { CK(cudaMemsetAsync(dst, 0, bytes, st)); });
}

// =================================================================================================
// weights
// =================================================================================================
struct HostW {
  std::map<std::string, std::vector<float>> t;
  std::map<std::string, std::vector<int64_t>> shape;
  const std::vector<float>& get(const std::string& k, std::initializer_list<int64_t> want) {
    auto it = t.find(k);
    if (it == t.end()) fail(AVC_ERR_WEIGHTS, "missing weight '%s'", k.c_str());
    const auto& s = shape[k];
    std::vector<int64_t> w(want);
    if (s != w) {
      std::string got, exp;
      for (auto v : s) got += std::to_string(v) + ",";
      for (auto v : w) exp += std::to_string(v) + ",";
      fail(AVC_ERR_WEIGHTS, "weight '%s' has shape [%s] expected [%s]", k.c_str(), got.c_str(), exp.c_str());
    }
    return it->second;
  }
};

// Conv1d weight [c_out][c_in][k] -> forward image [k][c_in][c_out'] and dgrad image [k rev][c_out'][c_in].
// `shuffle` > 1 permutes output channels so pixel_shuffle_1d becomes a reinterpretation of the row
// (n' = s*C + c  <->  n = shuffle*c + s).
ConvW pack_conv(avc_handle* h, HostW& hw, const std::string& key, int c_in, int c_out, int k, int stride, int shuffle) {
  const auto& w = hw.get(key + ".weight", {c_out, c_in, k});
  const auto& b = hw.get(key + ".bias", {c_out});
  ConvW c;
  c.c_in = c_in; c.c_out = c_out; c.k = k; c.stride = stride;
  std::vector<int> perm(c_out);
  const int C = c_out / shuffle;
  for (int np = 0; np < c_out; ++np) perm[np] = shuffle > 1 ? shuffle * (np % C) + np / C : np;
  std::vector<float> f((size_t)k * c_in * c_out), r((size_t)k * c_out * c_in), bb(c_out);
  for (int np = 0; np < c_out; ++np) {
    const int n = perm[np];
    bb[np] = b[n];
    for (int ci = 0; ci < c_in; ++ci)
      for (int j = 0; j < k; ++j) {
        const float v = w[((size_t)n * c_in + ci) * k + j];
        f[((size_t)j * c_in + ci) * c_out + np] = v;
        r[((size_t)(k - 1 - j) * c_out + np) * c_in + ci] = v;
      }
  }
  c.fwd = h->wmem.upload(f);
  c.bwd = h->wmem.upload(r);
  c.bias = h->wmem.upload(bb);
  if (k == 1 && c_in % 4 == 0 && c_out % 32 == 0) {
    // 3xTF32 planes of the [c_in][c_out] image: as a [rows = c_in][K = c_out] matrix it is the K-major weight operand of
    // this conv's dgrad (contract over c_out, produce c_in)
    std::vector<float> fh(f.size()), fl(f.size());
    for (size_t i = 0; i < f.size(); ++i) {
      uint32_t u;
      memcpy(&u, &f[i], 4);
      u = (u + 0x1000u) & 0xffffe000u;
      memcpy(&fh[i], &u, 4);
      fl[i] = f[i] - fh[i];
    }
    c.fwd_h = h->wmem.upload(fh);
    c.fwd_l = h->wmem.upload(fl);
  }
  tc_pack_both(h->wmem, c, f, r);     // B operand images for the tcgen05 path
  return c;
}

void pack_linear(avc_handle* h, HostW& hw, const std::string& key, int n_out, int n_in, float*& Wt, float*& W, float*& b) {
  const auto& w = hw.get(key + ".weight", {n_out, n_in});
  const auto& bb = hw.get(key + ".bias", {n_out});
  std::vector<float> t((size_t)n_in * n_out);
  for (int n = 0; n < n_out; ++n)
    for (int c = 0; c < n_in; ++c) t[(size_t)c * n_out + n] = w[(size_t)n * n_in + c];
  Wt = h->wmem.upload(t);
  W = h->wmem.upload(w);
  b = h->wmem.upload(bb);
}

void pack_encoder(avc_handle* h, HostW& hw, const std::string& pfx, EncoderW& E, const avc_encoder_desc& d, bool content) {
  E.d = d;
  E.n_bank = d.bank_size;
  E.c_cat = d.c_bank * E.n_bank + d.c_in;
  std::vector<float> bias_cat;
  for (int i = 0; i < E.n_bank; ++i) {
    E.bank[i] = pack_conv(h, hw, pfx + "conv_bank." + std::to_string(i), d.c_in, d.c_bank, i + 1, 1, 1);
    const auto& b = hw.get(pfx + "conv_bank." + std::to_string(i) + ".bias", {d.c_bank});
    bias_cat.insert(bias_cat.end(), b.begin(), b.end());
  }
  E.bank_bias = h->wmem.upload(bias_cat);
  E.in_conv = pack_conv(h, hw, pfx + "in_conv_layer", E.c_cat, d.c_h, 1, 1, 1);
  for (int l = 0; l < d.n_conv_blocks; ++l) {
    E.c1[l] = pack_conv(h, hw, pfx + "first_conv_layers." + std::to_string(l), d.c_h, d.c_h, d.kernel_size, 1, 1);
    E.c2[l] = pack_conv(h, hw, pfx + "second_conv_layers." + std::to_string(l), d.c_h, d.c_h, d.kernel_size, d.subsample[l], 1);
  }
  if (content) {
    E.mean_layer = pack_conv(h, hw, pfx + "mean_layer", d.c_h, d.c_out, 1, 1, 1);
  } else {
    for (int l = 0; l < d.n_dense_blocks; ++l) {
      pack_linear(h, hw, pfx + "first_dense_layers." + std::to_string(l), d.c_h, d.c_h, E.Wt1[l], E.W1[l], E.b1[l]);
      pack_linear(h, hw, pfx + "second_dense_layers." + std::to_string(l), d.c_h, d.c_h, E.Wt2[l], E.W2[l], E.b2[l]);
    }
    pack_linear(h, hw, pfx + "output_layer", d.c_out, d.c_h, E.Wto, E.Wo, E.bo);
  }
}

void pack_decoder(avc_handle* h, HostW& hw, const std::string& pfx, DecoderW& D, const avc_decoder_desc& d) {
  D.d = d;
  D.in_conv = pack_conv(h, hw, pfx + "in_conv_layer", d.c_in, d.c_h, 1, 1, 1);
  for (int l = 0; l < d.n_conv_blocks; ++l) {
    D.c1[l] = pack_conv(h, hw, pfx + "first_conv_layers." + std::to_string(l), d.c_h, d.c_h, d.kernel_size, 1, 1);
    D.c2[l] = pack_conv(h, hw, pfx + "second_conv_layers." + std::to_string(l), d.c_h, d.c_h * d.upsample[l], d.kernel_size, 1, d.upsample[l]);
  }
  for (int l = 0; l < 2 * d.n_conv_blocks; ++l)
    pack_linear(h, hw, pfx + "conv_affine_layers." + std::to_string(l), 2 * d.c_h, d.c_cond, D.aWt[l], D.aW[l], D.ab[l]);
  D.out_conv = pack_conv(h, hw, pfx + "out_conv_layer", d.c_h, d.c_out, 1, 1, 1);
}

void validate_desc(const avc_model_desc& m) {
  auto enc = [](const avc_encoder_desc& d, const char* nm, bool content) {
    if (d.c_in <= 0 || d.c_in % 4 || d.c_h != 128 || d.c_bank % 4 || d.c_bank > 128 || d.c_bank <= 0)
      fail(AVC_ERR_INVALID, "%s: need c_in %% 4 == 0, c_h == 128, c_bank %% 4 == 0 and <= 128", nm);
    if (d.c_in > 128) fail(AVC_ERR_INVALID, "%s: c_in > 128 unsupported", nm);
    if (d.bank_size < 1 || d.bank_size > AVC_MAX_BANK) fail(AVC_ERR_INVALID, "%s: bank_size must be 1..%d", nm, AVC_MAX_BANK);
    if (d.kernel_size < 1 || d.kernel_size > kMaxTaps) fail(AVC_ERR_INVALID, "%s: kernel_size must be 1..%d", nm, kMaxTaps);
    if (d.n_conv_blocks < 1 || d.n_conv_blocks > AVC_MAX_BLOCKS) fail(AVC_ERR_INVALID, "%s: n_conv_blocks must be 1..%d", nm, AVC_MAX_BLOCKS);
    for (int l = 0; l < d.n_conv_blocks; ++l)
      if (d.subsample[l] < 1 || d.subsample[l] > 4) fail(AVC_ERR_INVALID, "%s: subsample must be 1..4", nm);
    if ((d.c_bank * d.bank_size + d.c_in + 127) / 128 > kMaxGroups) fail(AVC_ERR_INVALID, "%s: bank concat too wide", nm);
    if (!content && (d.c_out != 128 || d.n_dense_blocks < 0 || d.n_dense_blocks > kTailMaxDense))
      fail(AVC_ERR_INVALID, "%s: need c_out == 128 and n_dense_blocks <= %d", nm, kTailMaxDense);
    if (content && (d.c_out % 4 || d.c_out > 128)) fail(AVC_ERR_INVALID, "%s: c_out must be a multiple of 4, <= 128", nm);
    if (d.neg_slope < 0.f || d.neg_slope >= 1.f) fail(AVC_ERR_INVALID, "%s: bad activation slope", nm);
  };
  enc(m.speaker, "SpeakerEncoder", false);
  enc(m.content, "ContentEncoder", true);
  const avc_decoder_desc& d = m.decoder;
  if (d.c_h != 128 || d.c_cond != 128 || d.c_in != m.content.c_out || d.c_out != m.speaker.c_in || d.c_in % 4)
    fail(AVC_ERR_INVALID, "Decoder: need c_h == c_cond == 128, c_in == content c_out, c_out == speaker c_in");
  if (d.n_conv_blocks < 1 || d.n_conv_blocks > AVC_MAX_BLOCKS) fail(AVC_ERR_INVALID, "Decoder: n_conv_blocks must be 1..%d", AVC_MAX_BLOCKS);
  if (d.kernel_size < 1 || d.kernel_size > kMaxTaps) fail(AVC_ERR_INVALID, "Decoder: kernel_size must be 1..%d", kMaxTaps);
  for (int l = 0; l < d.n_conv_blocks; ++l)
    if (d.upsample[l] < 1 || d.upsample[l] > 4) fail(AVC_ERR_INVALID, "Decoder: upsample must be 1..4");
  if (d.neg_slope < 0.f || d.neg_slope >= 1.f) fail(AVC_ERR_INVALID, "Decoder: bad activation slope");
}

// =================================================================================================
// attack plans
// =================================================================================================
enum AttackKind { K_EMB = 0, K_E2E = 1, K_FB = 2 };

int content_frames(const avc_handle* h, int T_src) {
  int t = T_src;
  for (int l = 0; l < h->desc.content.n_conv_blocks; ++l) t = cdiv(t, h->desc.content.subsample[l]);
  return t;
}
int decoder_frames(const avc_handle* h, int T_src) {
  int t = content_frames(h, T_src);
  for (int l = 0; l < h->desc.decoder.n_conv_blocks; ++l) t *= h->desc.decoder.upsample[l];
  return t;
}

void run_list(const std::vector<Launch>& v, cudaStream_t st) {
  for (const auto& l : v) l(st);
}

void check_strides(const int64_t s[3], const char* nm) {
  (void)s; (void)nm;   // any strides are legal; element (b,c,t) = base[b*s0 + c*s1 + t*s2]
}

// capture `reps` back-to-back iterations of the plan into a graph and instantiate it
void capture_iters(Plan& plan, int reps, cudaGraph_t* g, cudaGraphExec_t* x) {
  cudaStream_t cs;
  CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { cudaStreamDestroy(cs); fail(AVC_ERR_CUDA, "begin capture: %s", cudaGetErrorString(e)); }
  try {
    for (int r = 0; r < reps; ++r) run_list(plan.iter, cs);
  } catch (...) {
    cudaGraph_t bad = nullptr;
    cudaStreamEndCapture(cs, &bad);
    if (bad) cudaGraphDestroy(bad);
    cudaStreamDestroy(cs);
    throw;
  }
  e = cudaStreamEndCapture(cs, g);
  cudaStreamDestroy(cs);
  if (e != cudaSuccess) fail(AVC_ERR_CUDA, "end capture: %s", cudaGetErrorString(e));
  CK(cudaGraphInstantiate(x, *g, 0));
}

// Ragged batches (avc_attack_varlen): the perturbed utterances differ in length.  Only the speaker encoder on the perturbed
// batch (se1) sees them: its activations keep the padded layout [B, Tl[l], C] with Tl[l] the longest utterance's rows and
// a device table of every utterance's rows per level; rows past an utterance's length are dead -- no conv reads them for a
// live row or stores them, and the arena's zero-initialised slabs keep them 0 in the optimiser state and the perturbed
// input.  Every speaker-encoder conv of se1 runs on the tensor-core kernels, whatever its row count.
void check_ragged_lengths(const avc_handle* h, const std::vector<int>& frames) {
  for (size_t b = 0; b < frames.size(); ++b)
    if (frames[b] <= 0 || too_short_for_encoder(h->se, frames[b]))
      fail(AVC_ERR_INVALID, "utterance %zu of %d frames is too short for the speaker encoder's reflect padding", b, frames[b]);
}

// frames: per-utterance lengths of a ragged batch (a->vc_tgt, w0, adv_out, grad_out are then packed [sum T_b, C] and
// a->T_tgt is the longest), nullptr for equal lengths
std::unique_ptr<Plan> build_attack(avc_handle* h, AttackKind kind, const avc_attack_args* a, cudaStream_t st,
                                   const std::vector<int>* frames = nullptr) {
  if (!h->have_weights) fail(AVC_ERR_STATE, "avc_load_weights must be called before an attack");
  if (!a || !a->vc_tgt || !a->adv_tgt || !a->w0 || !a->adv_out) fail(AVC_ERR_INVALID, "null tensor argument");
  if (kind != K_EMB && !a->vc_src) fail(AVC_ERR_INVALID, "vc_src is required for e2e and fb attacks");
  if (a->B <= 0 || a->T_tgt <= 0 || a->T_adv <= 0 || a->n_iters < 0) fail(AVC_ERR_INVALID, "bad B/T/n_iters");
  const int B = a->B, T = a->T_tgt, C = h->desc.speaker.c_in;
  // provisioned iterations (Adam table, loss buffer): rounded up so that a cached plan serves later calls of the same shape
  const int n_iters = a->n_iters <= 64 ? 64 : (a->n_iters + 511) / 512 * 512;
  const float eps = a->eps;
  const EncoderW& SE = h->se;

  std::unique_ptr<Plan> plan_ptr(new Plan(&h->pool, st));
  Plan& plan = *plan_ptr;
  plan.n_iters = n_iters;
  plan.use_graph = a->use_graph != 0;
  plan.io.bind(*a);
  IoBind* io = &plan.io;
  Arena& m = plan.mem;
  Emitter S{h, &plan.setup, &plan.mem}, I{h, &plan.iter, &plan.mem}, F{h, &plan.finish, &plan.mem};

  // ---- state of the optimiser --------------------------------------------------------------
  const size_t nel = (size_t)B * T * C;
  float* x = m.f(nel);
  float* w = m.f(nel);
  float* mm = m.f(nel);
  float* vv = m.f(nel);
  float* gw = a->grad_out ? m.f(nel) : nullptr;
  int* step = m.raw<int>(1);
  unsigned int* done = m.raw<unsigned int>(1);
  std::vector<float> tab((size_t)std::max(n_iters, 1) * 2);
  for (int i = 0; i < n_iters; ++i) {   // torch/optim/adam.py: bias corrections in python floats (fp64)
    const double t = i + 1;
    const double bc1 = 1.0 - std::pow(0.9, t), bc2 = 1.0 - std::pow(0.999, t);
    tab[2 * i] = (float)(1e-3 / bc1);
    tab[2 * i + 1] = (float)std::sqrt(bc2);
  }
  float2* table = reinterpret_cast<float2*>(m.upload(tab));

  EncActs se1 = alloc_encoder(m, SE, B, T, true, false);
  const Tens adv = se1.input(SE);   // the perturbed utterance lives in the bank concat buffer
  Tens xT = tens(x, T, C), wT = tens(w, T, C);
  const bool ragged = frames != nullptr;
  const int* offs = nullptr;        // ragged: row offsets of the packed caller tensors, device [B+1]
  long long rows = (long long)B * T;
  if (ragged) {
    std::vector<int> o(B + 1, 0), len(frames->begin(), frames->end());
    for (int b = 0; b < B; ++b) o[b + 1] = o[b] + len[b];
    rows = o[B];
    offs = m.upload(o);
    for (int l = 0; l <= SE.d.n_conv_blocks; ++l) {
      se1.lens[l] = m.upload(len);
      if (l < SE.d.n_conv_blocks) for (int& t : len) t = cdiv(t, SE.d.subsample[l]);
    }
  }
  // the caller's utterance-shaped tensors: [B, C, T] strided, or packed [sum T_b, C] in a ragged batch
  auto utt_in = [&](Emitter& E, const float* const* src, const int64_t* s, const Tens& dst) {
    if (ragged) emit_layout_in_varlen_io(E, src, offs, dst, B, C, rows);
    else emit_layout_in_io(E, src, s, dst, B, C);
  };
  // a ragged batch takes the adversarial target through its own (equal-length) encoder pass even when T_adv == T_tgt
  const bool adv_in_se1 = !ragged && a->T_adv == T;
  {   // a (possibly reused) plan starts from a fresh optimiser: m = v = 0, step 0
    float* mz = mm; float* vz = vv; int* sz = step; unsigned int* dz = done;
    S.push(LK_COPY, 0, 8.0 * nel, [=](cudaStream_t s_) {
      CK(cudaMemsetAsync(mz, 0, nel * sizeof(float), s_)); CK(cudaMemsetAsync(vz, 0, nel * sizeof(float), s_));
      CK(cudaMemsetAsync(sz, 0, sizeof(int), s_)); CK(cudaMemsetAsync(dz, 0, sizeof(unsigned int), s_));
    });
  }
  utt_in(S, &io->vc_tgt, io->tgt_stride, xT);
  utt_in(S, &io->w0, io->w0_stride, wT);

  float* org = nullptr;   // targets
  float* tgt = nullptr;
  double inv_norm = a->inv_norm;
  int parts = B;
  float* loss_parts = nullptr;

  auto se_forward = [&](Emitter& E, const EncActs& A, int tail_mode, const float* tgt_e, const float* org_e,
                        float* emb_dst) {
    emit_bank_and_inconv(E, SE, A, false);
    emit_encoder_blocks_fwd(E, SE, A, false);
    TailArgs t = tail_args(SE, A);
    t.mode = tail_mode; t.tgt = tgt_e; t.org = org_e; t.inv_norm = (float)inv_norm; t.lam = 0.1f;
    t.loss_parts = loss_parts; t.step = step; t.parts_per_step = parts;
    if (emb_dst) t.emb = emb_dst;
    emit_tail(E, t, A.B);
  };
  auto perturb = [&](Emitter& E) {
    const unsigned g = ew_grid((long long)nel / 4, h->sm_count);
    E.push(LK_UPDATE, 0, 12.0 * nel, [=](cudaStream_t s_) { launch_k(perturb_kernel, g, 256, 0, s_, x, w, adv.p, adv.bs, adv.rs, B, T, C, eps); });
  };
  auto update = [&](Emitter& E, const Tens& gadv, const GradParts& gp) {
    UpdateArgs u{};
    u.n_gpart = gp.n;
    for (int q = 0; q < gp.n; ++q) u.g_part[q] = gp.p[q];
    u.g_adv = gadv.p; u.g_bs = gadv.bs; u.g_rs = gadv.rs; u.x = x; u.w = w; u.m = mm; u.v = vv;
    u.adv = adv.p; u.adv_bs = adv.bs; u.adv_rs = adv.rs; u.gw_out = gw; u.B = B; u.T = T; u.C = C; u.eps = eps;
    u.table = table; u.step = step; u.done = done;
    const unsigned g = ew_grid((long long)nel / 4, h->sm_count);
    E.push(LK_UPDATE, 0, 36.0 * nel, [=](cudaStream_t s_) { launch_k(adam_tanh_update_kernel, g, 256, 0, s_, u); });
  };

  if (kind == K_EMB) {
    if (inv_norm <= 0) inv_norm = 1.0 / ((double)B * SE.d.c_out);
    loss_parts = m.f((size_t)std::max(n_iters, 1) * parts);
    org = m.f((size_t)B * 128);
    tgt = m.f((size_t)B * 128);
    // targets (attack_utils.py:73-75)
    utt_in(S, &io->vc_tgt, io->tgt_stride, adv);
    se_forward(S, se1, TAIL_FWD, nullptr, nullptr, org);
    if (adv_in_se1) {
      emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, adv, B, C);
      se_forward(S, se1, TAIL_FWD, nullptr, nullptr, tgt);
    } else {
      EncActs seT = alloc_encoder(m, SE, B, a->T_adv, false, false);
      emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, seT.input(SE), B, C);
      se_forward(S, seT, TAIL_FWD, nullptr, nullptr, tgt);
    }
    perturb(S);
    // iteration (attack_utils.py:77-84)
    se_forward(I, se1, TAIL_FWD | TAIL_LOSS | TAIL_BWD, tgt, org, nullptr);
    Tens gin = tens(se1.gin, T, C);
    GradParts gp;
    emit_speaker_bwd(I, SE, se1, gin, &gp);
    update(I, gin, gp);
  } else {
    const int T_src = a->T_src;
    if (T_src <= 0) fail(AVC_ERR_INVALID, "bad T_src");
    const int L = content_frames(h, T_src), T_dec = decoder_frames(h, T_src), Cm = h->desc.decoder.c_out;
    // content code (loop invariant; the reference recomputes it every iteration, models.py:482)
    EncActs ce = alloc_encoder(m, h->ce, B, T_src, false, true);
    DecActs dec = alloc_decoder(m, h->dec, B, L, true);
    emit_layout_in_io(S, &io->vc_src, io->src_stride, ce.input(h->ce), B, C);
    emit_bank_and_inconv(S, h->ce, ce, true);
    emit_encoder_blocks_fwd(S, h->ce, ce, true);
    {
      const int nb = h->ce.d.n_conv_blocks;
      ConvArgs am = fwd_conv_args(h->ce.mean_layer, tens(ce.hout[nb - 1], L, h->ce.d.c_h), tens(dec.z, L, h->ce.d.c_out), B, false, 0.f);
      S.conv(am, &h->ce.mean_layer);
    }
    emit_decoder_const(S, h->dec, dec);

    if (kind == K_E2E) {
      const size_t nout = (size_t)B * T_dec * Cm;
      if (inv_norm <= 0) inv_norm = 1.0 / ((double)nout);
      float* dout = m.f(nout);
      float* gout = m.f(nout);
      org = m.f(nout);
      tgt = m.f(nout);
      Tens doutT = tens(dout, T_dec, Cm);
      const long long n4 = (long long)nout / 4;
      const unsigned mg = ew_grid(n4, h->sm_count);
      parts = (int)mg;
      loss_parts = m.f((size_t)std::max(n_iters, 1) * parts);
      // targets (attack_utils.py:35-37)
      utt_in(S, &io->vc_tgt, io->tgt_stride, adv);
      se_forward(S, se1, TAIL_FWD, nullptr, nullptr, nullptr);
      emit_decoder_fwd(S, h->dec, dec, se1.emb, doutT);
      emit_copy(S, org, dout, nout);
      if (adv_in_se1) {
        emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, adv, B, C);
        se_forward(S, se1, TAIL_FWD, nullptr, nullptr, nullptr);
        emit_decoder_fwd(S, h->dec, dec, se1.emb, doutT);
      } else {
        EncActs seT = alloc_encoder(m, SE, B, a->T_adv, false, false);
        emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, seT.input(SE), B, C);
        se_forward(S, seT, TAIL_FWD, nullptr, nullptr, nullptr);
        emit_decoder_fwd(S, h->dec, dec, seT.emb, doutT);
      }
      emit_copy(S, tgt, dout, nout);
      perturb(S);
      // iteration (attack_utils.py:39-46)
      se_forward(I, se1, TAIL_FWD, nullptr, nullptr, nullptr);
      emit_decoder_fwd(I, h->dec, dec, se1.emb, doutT);
      {
        const float invn = (float)inv_norm;
        float* lp = loss_parts; int* stp = step; const int pp = parts;
        I.push(LK_LOSS, 0, 16.0 * nout, [=](cudaStream_t s_) { launch_k(mse_grad_kernel, mg, 256, 0, s_, dout, tgt, org, gout, n4, invn, lp, stp, pp); });
      }
      emit_decoder_bwd(I, h->dec, dec, tens(gout, T_dec, Cm));
    } else {   // K_FB
      if (inv_norm <= 0) inv_norm = 1.0 / ((double)B * SE.d.c_out);
      loss_parts = m.f((size_t)std::max(n_iters, 1) * parts);
      org = m.f((size_t)B * 128);
      tgt = m.f((size_t)B * 128);
      EncActs se2 = alloc_encoder(m, SE, B, T_dec, true, false);   // speaker encoder on the converted utterance
      const Tens conv_out = se2.input(SE);
      // targets (attack_utils.py:117-119)
      utt_in(S, &io->vc_tgt, io->tgt_stride, adv);
      se_forward(S, se1, TAIL_FWD, nullptr, nullptr, nullptr);
      emit_decoder_fwd(S, h->dec, dec, se1.emb, conv_out);
      se_forward(S, se2, TAIL_FWD, nullptr, nullptr, org);
      if (adv_in_se1) {
        emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, adv, B, C);
        se_forward(S, se1, TAIL_FWD, nullptr, nullptr, tgt);
      } else {
        EncActs seT = alloc_encoder(m, SE, B, a->T_adv, false, false);
        emit_layout_in_io(S, &io->adv_tgt, io->adv_stride, seT.input(SE), B, C);
        se_forward(S, seT, TAIL_FWD, nullptr, nullptr, tgt);
      }
      perturb(S);
      // iteration (attack_utils.py:121-128)
      se_forward(I, se1, TAIL_FWD, nullptr, nullptr, nullptr);
      emit_decoder_fwd(I, h->dec, dec, se1.emb, conv_out);
      se_forward(I, se2, TAIL_FWD | TAIL_LOSS | TAIL_BWD, tgt, org, nullptr);
      Tens g2 = tens(se2.gin, T_dec, C);
      emit_speaker_bwd(I, SE, se2, g2);
      emit_decoder_bwd(I, h->dec, dec, g2);
    }
    // common tail of e2e / fb: d emb -> speaker encoder backward -> update
    {
      TailArgs t = tail_args(SE, se1);
      t.mode = TAIL_BWD; t.gemb = dec.gemb_parts; t.gemb_parts = 2 * dec.nb;
      emit_tail(I, t, B);
    }
    Tens gin = tens(se1.gin, T, C);
    GradParts gp;
    emit_speaker_bwd(I, SE, se1, gin, &gp);
    update(I, gin, gp);
  }

  // ---- finish: result, loss curve, last gradient -----------------------------------------------
  if (ragged) emit_layout_out_varlen_io(F, adv, offs, &io->adv_out, B, C, rows);
  else emit_layout_out_io(F, adv, &io->adv_out, io->out_stride, B, C);
  {
    float* lp = loss_parts; const int pp = parts;
    F.push(LK_LOSS, 0, 4.0 * pp * n_iters, [=](cudaStream_t s_) {
      const int n = io->n_iters;
      if (io->loss_out && n > 0) launch_k(loss_sum_kernel, (n + 127) / 128, 128, 0, s_, (const float*)lp, pp, n, io->loss_out);
    });
  }
  if (gw && ragged) {
    const Tens g = tens(gw, T, C);
    F.push(LK_LAYOUT, 0, 8.0 * rows * C, [=](cudaStream_t s_) {
      if (io->grad_out && io->n_iters > 0)
        launch_k(layout_out_varlen_kernel, dim3((unsigned)cdiv(T * C, 256), B), 256, 0, s_, (const float*)g.p, g.bs, g.rs, offs, io->grad_out, C);
    });
  } else if (gw) {
    const long long cs0 = (long long)C * T, cs1 = T;
    const Tens g = tens(gw, T, C);
    const long long n = (long long)B * T * C;
    F.push(LK_LAYOUT, 0, 8.0 * n, [=](cudaStream_t s_) {
      if (io->grad_out && io->n_iters > 0)
        launch_k(layout_out_kernel, (unsigned)((n + 255) / 256), 256, 0, s_, g.p, g.bs, g.rs, io->grad_out, cs0, cs1, 1LL, B, C, g.T);
    });
  }

  // ---- setup: targets, loop invariants, initial perturbation; then capture one iteration -----------
  // (arena zero fills / uploads are ordered on `st`: no device-wide synchronisation needed before the first launch)
  try {
    run_list(plan.setup, st);
    h->launches += (long long)plan.setup.size();
    h->launches_per_iter = (int)plan.iter.size();
    if (plan.use_graph) capture_iters(plan, 1, &plan.graph, &plan.exec);
  } catch (...) {
    cudaDeviceSynchronize();   // nothing may still be running when the arena is released
    throw;
  }
  return plan_ptr;
}

// ---- universal perturbation header (reference models/header_model.py:25-68; SURVEY 8f rank 2) --------
// speaker_encoder = this handle's AdaIN-VC SpeakerEncoder on mel.squeeze(1); source/target embeddings are loop
// invariants (the reference recomputes them every iteration, :48-49).  iter = forward, loss, backward and the
// batch-summed header gradient; iter2 = Adam + projection + next perturbed batch.
std::unique_ptr<Plan> build_header(avc_handle* h, const avc_header_args* a, cudaStream_t st) {
  if (!h->have_weights) fail(AVC_ERR_STATE, "avc_load_weights must be called before avc_header_*");
  if (!a || !a->source || !a->target || !a->header0 || !a->header_out) fail(AVC_ERR_INVALID, "null tensor argument");
  if (a->B <= 0 || a->T <= 0 || a->T_tgt <= 0 || a->n_iters < 0 || a->lr <= 0.f) fail(AVC_ERR_INVALID, "bad B/T/n_iters/lr");
  const int B = a->B, T = a->T, C = h->desc.speaker.c_in, n_iters = a->n_iters;
  const EncoderW& SE = h->se;
  std::unique_ptr<Plan> plan_ptr(new Plan(&h->pool, st));
  Plan& plan = *plan_ptr;
  plan.n_iters = n_iters;
  plan.use_graph = a->use_graph != 0;
  Arena& m = plan.mem;
  Emitter S{h, &plan.setup, &plan.mem}, I{h, &plan.iter, &plan.mem}, F{h, &plan.finish, &plan.mem};
  const size_t nel = (size_t)B * T * C, nh = (size_t)T * C;
  float* x = m.f(nel);
  float* hdr = m.f(nh);
  float* mm = m.f(nh);
  float* vv = m.f(nh);
  float* gh = m.f(nh);
  plan.gh = gh; plan.gh_n = (long long)nh;
  int* step = m.raw<int>(1);
  unsigned int* done = m.raw<unsigned int>(1);
  std::vector<float> tab((size_t)std::max(n_iters, 1) * 2);
  for (int i = 0; i < n_iters; ++i) {
    const double t = i + 1;
    tab[2 * i] = (float)((double)a->lr / (1.0 - std::pow(0.9, t)));
    tab[2 * i + 1] = (float)std::sqrt(1.0 - std::pow(0.999, t));
  }
  float2* table = reinterpret_cast<float2*>(m.upload(tab));
  EncActs se1 = alloc_encoder(m, SE, B, T, true, false);
  const Tens adv = se1.input(SE);
  emit_layout_in(S, a->source, a->src_stride, tens(x, T, C), B, C);
  const int64_t hs[3] = {0, a->hdr_stride[0], a->hdr_stride[1]};
  emit_layout_in(S, a->header0, hs, tens(hdr, T, C), 1, C);
  const double inv_norm = a->inv_norm > 0 ? a->inv_norm : 1.0 / ((double)B * SE.d.c_out);
  const int parts = B;
  float* loss_parts = m.f((size_t)std::max(n_iters, 1) * parts);
  float* org = m.f((size_t)B * 128);
  float* tgt = m.f((size_t)B * 128);
  auto se_forward = [&](Emitter& E, const EncActs& A, int tail_mode, const float* tgt_e, const float* org_e, float* emb_dst) {
    emit_bank_and_inconv(E, SE, A, false);
    emit_encoder_blocks_fwd(E, SE, A, false);
    TailArgs t = tail_args(SE, A);
    t.mode = tail_mode; t.tgt = tgt_e; t.org = org_e; t.inv_norm = (float)inv_norm; t.lam = a->lambda;
    t.loss_parts = loss_parts; t.step = step; t.parts_per_step = parts;
    if (emb_dst) t.emb = emb_dst;
    emit_tail(E, t, A.B);
  };
  // loop invariants: embeddings of the clean source and of the target (header_model.py:48-49)
  emit_layout_in(S, a->source, a->src_stride, adv, B, C);
  se_forward(S, se1, TAIL_FWD, nullptr, nullptr, org);
  if (a->T_tgt == T) {
    emit_layout_in(S, a->target, a->tgt_stride, adv, B, C);
    se_forward(S, se1, TAIL_FWD, nullptr, nullptr, tgt);
  } else {
    EncActs seT = alloc_encoder(m, SE, B, a->T_tgt, false, false);
    emit_layout_in(S, a->target, a->tgt_stride, seT.input(SE), B, C);
    se_forward(S, seT, TAIL_FWD, nullptr, nullptr, tgt);
  }
  const unsigned gp = ew_grid((long long)nel / 4, h->sm_count), gt = ew_grid((long long)nh / 4, h->sm_count);
  S.push(LK_UPDATE, 0, 8.0 * nel, [=](cudaStream_t s_) { launch_k(header_perturb_kernel, gp, 256, 0, s_, (const float*)x, (const float*)hdr, adv.p, adv.bs, adv.rs, B, T, C); });
  // iteration, gradient half
  se_forward(I, se1, TAIL_FWD | TAIL_LOSS | TAIL_BWD, tgt, org, nullptr);
  Tens gin = tens(se1.gin, T, C);
  GradParts gparts;
  emit_speaker_bwd(I, SE, se1, gin, &gparts);
  I.push(LK_UPDATE, 0, 8.0 * nel, [=](cudaStream_t s_) { launch_k(header_grad_kernel, gt, 256, 0, s_, (const float*)gin.p, gin.bs, gin.rs, gparts.p[0], gparts.p[1], (const float*)x, (const float*)hdr, gh, B, T, C); });
  // iteration, apply half
  {
    HeaderApplyArgs u{};
    u.gh = gh; u.h = hdr; u.m = mm; u.v = vv; u.x = x; u.adv = adv.p; u.adv_bs = adv.bs; u.adv_rs = adv.rs;
    u.B = B; u.T = T; u.C = C; u.eps = a->eps; u.table = table; u.step = step; u.done = done;
    Emitter I2{h, &plan.iter2, &plan.mem};
    I2.push(LK_UPDATE, 0, 8.0 * nel + 28.0 * nh, [=](cudaStream_t s_) { launch_k(header_apply_kernel, gt, 256, 0, s_, u); });
  }
  // finish: header, loss curve, last gradient
  {
    const int64_t os[3] = {0, a->out_stride[0], a->out_stride[1]};
    emit_layout_out(F, tens(hdr, T, C), a->header_out, os, 1, C);
  }
  if (a->loss_out && n_iters > 0) {
    float* lp = loss_parts; float* lo = a->loss_out; const int pp = parts;
    F.push(LK_LOSS, 0, 4.0 * pp * n_iters, [=](cudaStream_t s_) { launch_k(loss_sum_kernel, (n_iters + 127) / 128, 128, 0, s_, (const float*)lp, pp, n_iters, lo); });
  }
  if (a->grad_out && n_iters > 0) {
    const int64_t cs[3] = {0, (int64_t)T, 1};
    emit_layout_out(F, tens(gh, T, C), a->grad_out, cs, 1, C);
  }
  CK(cudaDeviceSynchronize());
  try {
    run_list(plan.setup, st);
    h->launches += (long long)plan.setup.size();
    h->launches_per_iter = (int)(plan.iter.size() + plan.iter2.size());
    if (n_iters > 0 && plan.use_graph) {
      auto capture = [&](const std::vector<Launch>& v, cudaGraph_t* g, cudaGraphExec_t* xg) {
        cudaStream_t cs;
        CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) { cudaStreamDestroy(cs); fail(AVC_ERR_CUDA, "begin capture: %s", cudaGetErrorString(e)); }
        try { run_list(v, cs); } catch (...) { cudaGraph_t bad = nullptr; cudaStreamEndCapture(cs, &bad); if (bad) cudaGraphDestroy(bad); cudaStreamDestroy(cs); throw; }
        e = cudaStreamEndCapture(cs, g);
        cudaStreamDestroy(cs);
        if (e != cudaSuccess) fail(AVC_ERR_CUDA, "end capture: %s", cudaGetErrorString(e));
        CK(cudaGraphInstantiate(xg, *g, 0));
      };
      capture(plan.iter, &plan.graph, &plan.exec);
      capture(plan.iter2, &plan.graph2, &plan.exec2);
    }
  } catch (...) {
    cudaDeviceSynchronize();
    throw;
  }
  return plan_ptr;
}

// ---- speaker-embedding loss gradient service (reference train_predictive.py:113-123; SURVEY 8f rank 3) -------
// iter = embeddings of the clean source and of the target (forward only), then forward / loss / backward of the perturbed
// batch and the input gradient in the caller's layout.  Every launch reads the caller's buffers at run time: one
// captured graph serves every training step.
std::unique_ptr<Plan> build_spkgrad(avc_handle* h, const avc_spk_grad_args* a, cudaStream_t st) {
  if (!h->have_weights) fail(AVC_ERR_STATE, "avc_load_weights must be called before avc_spk_grad_*");
  if (!a || !a->perturbed || !a->source || !a->target || !a->grad_out) fail(AVC_ERR_INVALID, "null tensor argument");
  if (a->B <= 0 || a->T <= 0 || a->T_tgt <= 0) fail(AVC_ERR_INVALID, "bad B/T");
  check_strides(a->p_stride, "perturbed"); check_strides(a->s_stride, "source"); check_strides(a->t_stride, "target");
  check_strides(a->g_stride, "grad_out");
  const int B = a->B, T = a->T, C = h->desc.speaker.c_in;
  const EncoderW& SE = h->se;
  std::unique_ptr<Plan> plan_ptr(new Plan(&h->pool, st));
  Plan& plan = *plan_ptr;
  plan.n_iters = 1 << 30;
  plan.io.n_iters = 1 << 30;
  plan.use_graph = a->use_graph != 0;
  Arena& m = plan.mem;
  Emitter I{h, &plan.iter, &plan.mem};
  const size_t nel = (size_t)B * T * C;
  int* step = m.raw<int>(1);              // stays 0: one loss slot per utterance, overwritten every step
  const double inv_norm = a->inv_norm > 0 ? a->inv_norm : 1.0 / ((double)B * SE.d.c_out);
  const int parts = B;
  float* loss_parts = m.f((size_t)parts);
  float* org = m.f((size_t)2 * B * 128);       // org | tgt adjacent ([2B,128]): the 2B-utterance tail writes both
  float* tgt = org + (size_t)B * 128;
  const float lam = a->lambda;
  EncActs se1;
  if (a->T_tgt == T) {
    // equal lengths (the trainer's case): ONE forward pass over [perturbed; source; target] -- 3B utterances fill the
    // tensor-core tiles better than three passes of B -- then the dense tail forward on the last 2B utterances and
    // forward + loss + backward on the first B.  Every buffer is batch-major, so the first B utterances of the 3B
    // activations ARE the activations the backward pass needs.
    EncActs se3 = alloc_encoder(m, SE, 3 * B, T, false, false);
    const int ch = SE.d.c_h;
    se3.gA = m.f((size_t)B * T * ch); se3.gB = m.f((size_t)B * T * ch); se3.gH = m.f((size_t)B * T * ch);
    se3.gcat = m.f((size_t)B * T * SE.c_cat); se3.gin = m.f((size_t)B * T * SE.d.c_in);
    Tens in = se3.input(SE);
    emit_layout_in(I, a->perturbed, a->p_stride, in, B, C);
    in.p += (long long)B * in.bs;
    emit_layout_in(I, a->source, a->s_stride, in, B, C);
    in.p += (long long)B * in.bs;
    emit_layout_in(I, a->target, a->t_stride, in, B, C);
    emit_bank_and_inconv(I, SE, se3, false);
    emit_encoder_blocks_fwd(I, SE, se3, false);
    {   // embeddings of source (-> org) and target (-> tgt): utterances [B, 3B)
      TailArgs t = tail_args(SE, se3);
      t.h += (long long)B * t.h_bs;
      t.acts += (size_t)B * (3 * SE.d.n_dense_blocks + 1) * 128;
      t.gpool += (size_t)B * 128;
      t.mode = TAIL_FWD; t.inv_norm = (float)inv_norm; t.lam = lam;
      t.loss_parts = loss_parts; t.step = step; t.parts_per_step = parts;
      t.emb = org;                      // org [B,128] and tgt [B,128] are adjacent: one [2B,128] block
      emit_tail(I, t, 2 * B);
    }
    se1 = se3; se1.B = B;
    {
      TailArgs t = tail_args(SE, se1);
      t.mode = TAIL_FWD | TAIL_LOSS | TAIL_BWD; t.tgt = tgt; t.org = org; t.inv_norm = (float)inv_norm; t.lam = lam;
      t.loss_parts = loss_parts; t.step = step; t.parts_per_step = parts;
      emit_tail(I, t, B);
    }
  } else {
    se1 = alloc_encoder(m, SE, B, T, true, false);
    const Tens adv = se1.input(SE);
    auto se_forward = [&](const EncActs& A, int tail_mode, const float* tgt_e, const float* org_e, float* emb_dst) {
      emit_bank_and_inconv(I, SE, A, false);
      emit_encoder_blocks_fwd(I, SE, A, false);
      TailArgs t = tail_args(SE, A);
      t.mode = tail_mode; t.tgt = tgt_e; t.org = org_e; t.inv_norm = (float)inv_norm; t.lam = lam;
      t.loss_parts = loss_parts; t.step = step; t.parts_per_step = parts;
      if (emb_dst) t.emb = emb_dst;
      emit_tail(I, t, A.B);
    };
    emit_layout_in(I, a->source, a->s_stride, adv, B, C);
    se_forward(se1, TAIL_FWD, nullptr, nullptr, org);
    EncActs seT = alloc_encoder(m, SE, B, a->T_tgt, false, false);
    emit_layout_in(I, a->target, a->t_stride, seT.input(SE), B, C);
    se_forward(seT, TAIL_FWD, nullptr, nullptr, tgt);
    emit_layout_in(I, a->perturbed, a->p_stride, adv, B, C);
    se_forward(se1, TAIL_FWD | TAIL_LOSS | TAIL_BWD, tgt, org, nullptr);
  }
  Tens gin = tens(se1.gin, T, C);
  GradParts gparts;
  emit_speaker_bwd(I, SE, se1, gin, &gparts);
  {
    const unsigned g = ew_grid((long long)nel, h->sm_count);
    float* dst = a->grad_out;
    const long long sb = a->g_stride[0], sc = a->g_stride[1], stt = a->g_stride[2];
    I.push(LK_LAYOUT, 0, 8.0 * nel, [=](cudaStream_t s_) { launch_k(spk_grad_out_kernel, g, 256, 0, s_, (const float*)gin.p, gin.bs, gin.rs, gparts.p[0], gparts.p[1], dst, sb, sc, stt, B, T, C); });
  }
  if (a->loss_out) {
    float* lo = a->loss_out;
    I.push(LK_LOSS, 0, 4.0 * parts, [=](cudaStream_t s_) { launch_k(loss_sum_kernel, 1, 128, 0, s_, (const float*)loss_parts, parts, 1, lo); });
  }
  CK(cudaStreamSynchronize(st));
  h->launches_per_iter = (int)plan.iter.size();
  if (plan.use_graph) capture_iters(plan, 1, &plan.graph, &plan.exec);
  return plan_ptr;
}

// phase 0: n whole iterations; 1: the gradient half of ONE iteration; 2: the apply half of ONE iteration
void step_header(avc_handle* h, Plan& plan, int n, int phase, cudaStream_t st) {
  if (plan.finished) fail(AVC_ERR_STATE, "session already finished");
  if (plan.iter2.empty()) fail(AVC_ERR_STATE, "not a header-optimisation session");
  if (phase < 0 || phase > 2 || n < 0) fail(AVC_ERR_INVALID, "bad phase / count");
  const int iters = phase == 0 ? n : (phase == 2 ? 1 : 0);
  if (plan.done_iters + iters > plan.n_iters) fail(AVC_ERR_INVALID, "session was opened for %d iterations, %d done", plan.n_iters, plan.done_iters);
  auto half = [&](const std::vector<Launch>& v, cudaGraphExec_t x) { if (x) CK(cudaGraphLaunch(x, st)); else run_list(v, st); };
  try {
    if (phase == 0) for (int i = 0; i < n; ++i) { half(plan.iter, plan.exec); half(plan.iter2, plan.exec2); }
    else if (phase == 1) half(plan.iter, plan.exec);
    else half(plan.iter2, plan.exec2);
  } catch (...) {
    cudaDeviceSynchronize();
    throw;
  }
  plan.done_iters += iters;
  h->launches += (long long)(phase == 0 ? (plan.iter.size() + plan.iter2.size()) * n : (phase == 1 ? plan.iter.size() : plan.iter2.size()));
}

void step_attack(avc_handle* h, Plan& plan, int n, cudaStream_t st) {
  if (plan.finished) fail(AVC_ERR_STATE, "attack session already finished");
  if (n < 0 || plan.done_iters + n > plan.io.n_iters)
    fail(AVC_ERR_INVALID, "session was opened for %d iterations, %d done, %d more requested", plan.io.n_iters, plan.done_iters, n);
  // kUnroll iterations per graph launch, captured the first time a call is long enough to profit from it
  if (plan.exec && !plan.execU && n >= 2 * kUnroll) capture_iters(plan, kUnroll, &plan.graphU, &plan.execU);
  try {
    if (plan.exec) {
      int left = n;
      if (plan.execU) for (; left >= kUnroll; left -= kUnroll) CK(cudaGraphLaunch(plan.execU, st));
      for (; left > 0; --left) CK(cudaGraphLaunch(plan.exec, st));
    } else {
      for (int i = 0; i < n; ++i) run_list(plan.iter, st);
    }
  } catch (...) {
    cudaDeviceSynchronize();
    throw;
  }
  plan.done_iters += n;
  h->launches += (long long)plan.iter.size() * n;
}

void finish_attack(avc_handle* h, Plan& plan, cudaStream_t st) {
  if (plan.finished) return;
  plan.finished = true;
  try {
    run_list(plan.finish, st);
    h->launches += (long long)plan.finish.size();
    CK(cudaStreamSynchronize(st));   // the session's buffers are freed next
  } catch (...) {
    cudaDeviceSynchronize();
    throw;
  }
}

// ---- plan cache ------------------------------------------------------------------------------------------
PlanKey make_key(const avc_handle* h, int kind, const avc_attack_args* a, const std::vector<int>* frames) {
  PlanKey k;
  if (!a) return k;
  if (frames) k.frames = *frames;
  k.kind = kind; k.B = a->B; k.T_tgt = a->T_tgt; k.T_adv = a->T_adv; k.T_src = kind == K_EMB ? 0 : a->T_src;
  k.use_graph = a->use_graph != 0; k.has_grad = a->grad_out != nullptr; k.conv_impl = h->conv_impl; k.tc_min_rows = h->tc_min_rows;
  k.eps = a->eps; k.inv_norm = a->inv_norm > 0 ? a->inv_norm : 0.0;
  return k;
}
constexpr size_t kPlanCacheMaxBytes = 512ull << 20;   // batch-1 .. batch-32 plans; the multi-GB batched plans are rebuilt
constexpr size_t kPlanCacheEntries = 4;

std::unique_ptr<Plan> take_cached(avc_handle* h, const PlanKey& key, int n_iters) {
  static const bool off = getenv("AVC_NO_PLAN_CACHE") != nullptr;
  if (off) return nullptr;
  for (size_t i = 0; i < h->plan_cache.size(); ++i)
    if (h->plan_cache[i]->key == key && h->plan_cache[i]->n_iters >= n_iters) {
      std::unique_ptr<Plan> p = std::move(h->plan_cache[i]);
      h->plan_cache.erase(h->plan_cache.begin() + i);
      ++h->plan_cache_hits;
      return p;
    }
  return nullptr;
}
void put_cached(avc_handle* h, std::unique_ptr<Plan> plan) {
  if (!plan || plan->key.kind < 0 || plan->mem.bytes > kPlanCacheMaxBytes) return;   // dropped: buffers go back to the slab pool
  for (auto& q : h->plan_cache) if (q->key == plan->key && q->n_iters >= plan->n_iters) return;
  h->plan_cache.push_back(std::move(plan));
  if (h->plan_cache.size() > kPlanCacheEntries) h->plan_cache.erase(h->plan_cache.begin());
}

// a plan ready to iterate: a cached one rebound to this call's tensors (its setup re-run), else a new one
std::unique_ptr<Plan> acquire_attack(avc_handle* h, AttackKind kind, const avc_attack_args* a, cudaStream_t st,
                                     const std::vector<int>* frames = nullptr) {
  PlanKey key = make_key(h, (int)kind, a, frames);
  std::unique_ptr<Plan> plan = a ? take_cached(h, key, a->n_iters) : nullptr;
  if (plan) {
    if (!a->vc_tgt || !a->adv_tgt || !a->w0 || !a->adv_out || (kind != K_EMB && !a->vc_src)) fail(AVC_ERR_INVALID, "null tensor argument");
    plan->io.bind(*a);
    plan->done_iters = 0;
    plan->finished = false;
    try {
      run_list(plan->setup, st);
    } catch (...) {
      cudaDeviceSynchronize();
      throw;
    }
    h->launches += (long long)plan->setup.size();
    h->launches_per_iter = (int)plan->iter.size();
    return plan;
  }
  plan = build_attack(h, kind, a, st, frames);
  plan->key = std::move(key);
  return plan;
}

void run_attack(avc_handle* h, AttackKind kind, const avc_attack_args* a, cudaStream_t st, const std::vector<int>* frames = nullptr) {
  static const bool timing = getenv("AVC_TIMING") != nullptr;   // host-side phase times on stderr
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  const long long hits0 = h->plan_cache_hits;
  std::unique_ptr<Plan> plan = acquire_attack(h, kind, a, st, frames);
  const double t1 = now();
  step_attack(h, *plan, a->n_iters, st);
  const double t2 = now();
  finish_attack(h, *plan, st);
  const double t3 = now();
  put_cached(h, std::move(plan));
  if (timing) fprintf(stderr, "[avc] attack kind %d: %s %.2f ms, enqueue %.2f ms, drain+finish %.2f ms, release %.2f ms\n", (int)kind,
                      h->plan_cache_hits > hits0 ? "rebind" : "build", t1 - t0, t2 - t1, t3 - t2, now() - t3);
}

template <class Fn>
int guarded(avc_handle* h, Fn&& fn) {
  try {
    DeviceGuard dg(h ? h->device : -1);
    fn();
    return AVC_OK;
  } catch (const Fail& f) {
    if (h) h->err = f.msg; else g_create_error = f.msg;
    return f.code;
  } catch (const std::exception& e) {
    if (h) h->err = e.what(); else g_create_error = e.what();
    return AVC_ERR_INVALID;
  }
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
namespace {
// run a unit entry point's launches; with avc_unit_timing set, repeat them and keep the device time of one repetition
template <class F>
void run_unit(avc_handle* h, cudaStream_t st, F&& run) {
  run();
  h->launches += 1;
  if (h->unit_reps > 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, st));
    for (int r = 0; r < h->unit_reps; ++r) run();
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    h->unit_ms = ms / (float)h->unit_reps;
    h->launches += h->unit_reps;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  CK(cudaStreamSynchronize(st));
}
}  // namespace

extern "C" {

#ifndef AVC_SRC_HASH
#define AVC_SRC_HASH "unhashed-build!!"
#endif
// "... src <16 hex digits>": sha256 prefix of the sources this binary was compiled from (attack_vc_b200/build.py)
const char* avc_version(void) { return "avc_b200 0.2 (sm_100a) src " AVC_SRC_HASH; }

int avc_create(avc_handle** out, const avc_model_desc* desc, int device) {
  if (!out || !desc) { g_create_error = "null argument"; return AVC_ERR_INVALID; }
  *out = nullptr;
  return guarded(nullptr, [&] {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) fail(AVC_ERR_CUDA, "no CUDA device available (%s); libavc_b200 has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= n) fail(AVC_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    validate_desc(*desc);
    DeviceGuard dg(device);
    cudaDeviceProp p{};
    CK(cudaGetDeviceProperties(&p, device));
    if (p.major < 10) fail(AVC_ERR_CUDA, "device %d is sm_%d%d; libavc_b200 is built for sm_100a only", device, p.major, p.minor);
    auto h = std::make_unique<avc_handle>();
    h->device = device;
    h->sm_count = p.multiProcessorCount;
    h->desc = *desc;
    if (const char* s = getenv("AVC_CONV_IMPL")) h->conv_impl = atoi(s);
    if (const char* s = getenv("AVC_TC_MIN_ROWS")) h->tc_min_rows = atoll(s);
    init_kernel_attributes();
    *out = h.release();
  });
}

void avc_destroy(avc_handle* h) {
  if (!h) return;
  DeviceGuard dg(h->device);
  cudaDeviceSynchronize();
  delete h;
}

const char* avc_last_error(const avc_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int avc_load_weights(avc_handle* h, const avc_weight_view* tensors, int32_t n) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!tensors || n <= 0) fail(AVC_ERR_INVALID, "no tensors");
    HostW hw;
    for (int i = 0; i < n; ++i) {
      const avc_weight_view& v = tensors[i];
      if (!v.name || !v.data || v.ndim < 1 || v.ndim > 4) fail(AVC_ERR_WEIGHTS, "bad weight view %d", i);
      size_t cnt = 1;
      std::vector<int64_t> shp;
      for (int d = 0; d < v.ndim; ++d) { cnt *= (size_t)v.shape[d]; shp.push_back(v.shape[d]); }
      std::vector<float> host(cnt);
      CK(cudaMemcpy(host.data(), v.data, cnt * sizeof(float), cudaMemcpyDeviceToHost));
      hw.t[v.name] = std::move(host);
      hw.shape[v.name] = shp;
    }
    if (h->have_weights) fail(AVC_ERR_STATE, "weights already loaded; create a new handle");
    pack_encoder(h, hw, "speaker_encoder.", h->se, h->desc.speaker, false);
    pack_encoder(h, hw, "content_encoder.", h->ce, h->desc.content, true);
    pack_decoder(h, hw, "decoder.", h->dec, h->desc.decoder);
    CK(cudaDeviceSynchronize());
    h->have_weights = true;
  });
}

int avc_emb_attack(avc_handle* h, const avc_attack_args* a, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] { run_attack(h, K_EMB, a, (cudaStream_t)stream); });
}
int avc_e2e_attack(avc_handle* h, const avc_attack_args* a, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] { run_attack(h, K_E2E, a, (cudaStream_t)stream); });
}
int avc_fb_attack(avc_handle* h, const avc_attack_args* a, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] { run_attack(h, K_FB, a, (cudaStream_t)stream); });
}

int avc_attack_varlen(avc_handle* h, int32_t kind, const avc_attack_varlen_args* v, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (kind < 0 || kind > 2) fail(AVC_ERR_INVALID, "kind must be 0 (emb), 1 (e2e) or 2 (fb)");
    if (!v || !v->frames_host || v->B <= 0) fail(AVC_ERR_INVALID, "null argument or B <= 0");
    if (h->conv_impl == 1 || h->conv_impl == 3)
      fail(AVC_ERR_INVALID, "ragged attacks run on the tensor-core kernels (AVC_CONV_IMPL=%d selects the CUDA cores)", h->conv_impl);
    std::vector<int> frames(v->frames_host, v->frames_host + v->B);
    check_ragged_lengths(h, frames);
    avc_attack_args a{};
    a.vc_tgt = v->vc_tgt; a.B = v->B; a.T_tgt = *std::max_element(frames.begin(), frames.end());
    a.adv_tgt = v->adv_tgt; a.T_adv = v->T_adv;
    a.vc_src = v->vc_src; a.T_src = v->T_src;
    for (int i = 0; i < 3; ++i) { a.adv_stride[i] = v->adv_stride[i]; a.src_stride[i] = v->src_stride[i]; }
    a.w0 = v->w0; a.adv_out = v->adv_out; a.loss_out = v->loss_out; a.grad_out = v->grad_out;
    a.eps = v->eps; a.n_iters = v->n_iters; a.inv_norm = v->inv_norm; a.use_graph = v->use_graph;
    run_attack(h, (AttackKind)kind, &a, (cudaStream_t)stream, &frames);
  });
}

int avc_attack_begin(avc_handle* h, int32_t kind, const avc_attack_args* a, void* stream, avc_session** out) {
  if (!h || !out) return AVC_ERR_INVALID;
  *out = nullptr;
  return guarded(h, [&] {
    if (kind < 0 || kind > 2) fail(AVC_ERR_INVALID, "kind must be 0 (emb), 1 (e2e) or 2 (fb)");
    std::unique_ptr<Plan> plan = acquire_attack(h, (AttackKind)kind, a, (cudaStream_t)stream);
    avc_session* s = new avc_session{h, std::move(plan)};
    *out = s;
  });
}

int avc_attack_step(avc_session* s, int32_t n, void* stream) {
  if (!s) return AVC_ERR_INVALID;
  return guarded(s->h, [&] { step_attack(s->h, *s->plan, n, (cudaStream_t)stream); });
}

int avc_attack_end(avc_session* s, void* stream) {
  if (!s) return AVC_ERR_INVALID;
  int rc = guarded(s->h, [&] { finish_attack(s->h, *s->plan, (cudaStream_t)stream); });
  DeviceGuard dg(s->h->device);
  cudaDeviceSynchronize();
  if (rc == AVC_OK) put_cached(s->h, std::move(s->plan));   // idle now: the next call of this shape rebinds it
  delete s;
  return rc;
}

int avc_header_begin(avc_handle* h, const avc_header_args* a, void* stream, avc_session** out) {
  if (!h || !out) return AVC_ERR_INVALID;
  *out = nullptr;
  return guarded(h, [&] {
    std::unique_ptr<Plan> plan = build_header(h, a, (cudaStream_t)stream);
    *out = new avc_session{h, std::move(plan)};
  });
}

int avc_header_step(avc_session* s, int32_t n, int32_t phase, void* stream) {
  if (!s) return AVC_ERR_INVALID;
  return guarded(s->h, [&] { step_header(s->h, *s->plan, n, phase, (cudaStream_t)stream); });
}

int avc_spk_grad_begin(avc_handle* h, const avc_spk_grad_args* a, void* stream, avc_session** out) {
  if (!h || !out) return AVC_ERR_INVALID;
  *out = nullptr;
  return guarded(h, [&] {
    std::unique_ptr<Plan> plan = build_spkgrad(h, a, (cudaStream_t)stream);
    *out = new avc_session{h, std::move(plan)};
  });
}

int avc_spk_grad_step(avc_session* s, void* stream) {
  if (!s) return AVC_ERR_INVALID;
  return guarded(s->h, [&] {
    if (!s->plan->iter2.empty() || !s->plan->setup.empty()) fail(AVC_ERR_STATE, "not a speaker-gradient session");
    step_attack(s->h, *s->plan, 1, (cudaStream_t)stream);
  });
}

float* avc_header_grad_buffer(avc_session* s, int64_t* n) {
  if (!s || !s->plan->gh) return nullptr;
  if (n) *n = s->plan->gh_n;
  return s->plan->gh;
}

int avc_header_optimize(avc_handle* h, const avc_header_args* a, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    std::unique_ptr<Plan> plan = build_header(h, a, (cudaStream_t)stream);
    step_header(h, *plan, a->n_iters, 0, (cudaStream_t)stream);
    finish_attack(h, *plan, (cudaStream_t)stream);
  });
}

int32_t avc_session_launches(const avc_session* s) { return s ? (int32_t)s->plan->iter.size() : -1; }

// Run ONE iteration eagerly with a CUDA event pair around every launch (stream-ordered, so each
// kernel is timed in isolation).  Counts as one of the session's iterations.
int avc_session_profile(avc_session* s, int32_t cap, int32_t* kind, float* ms, double* flops, double* bytes, void* stream) {
  if (!s) return AVC_ERR_INVALID;
  return guarded(s->h, [&] {
    Plan& plan = *s->plan;
    const int n = (int)plan.iter.size();
    if (cap < n || !kind || !ms || !flops || !bytes) fail(AVC_ERR_INVALID, "profile arrays must hold %d entries", n);
    if (plan.finished || plan.done_iters + 1 > (plan.key.kind >= 0 ? plan.io.n_iters : plan.n_iters)) fail(AVC_ERR_STATE, "no iteration left to profile");
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CK(cudaEventCreate(&e));
    try {
      CK(cudaEventRecord(ev[0], st));
      for (int i = 0; i < n; ++i) {
        plan.iter[i](st);
        CK(cudaEventRecord(ev[i + 1], st));
      }
      CK(cudaStreamSynchronize(st));
    } catch (...) {
      cudaDeviceSynchronize();
      for (auto& e : ev) cudaEventDestroy(e);
      throw;
    }
    for (int i = 0; i < n; ++i) {
      CK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
      kind[i] = plan.iter[i].kind; flops[i] = plan.iter[i].flops; bytes[i] = plan.iter[i].bytes;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    plan.done_iters += 1;
    s->h->launches += n;
  });
}

int32_t avc_decoder_frames(const avc_handle* h, int32_t T_src) { return h ? decoder_frames(h, T_src) : -1; }

int avc_speaker_encoder(avc_handle* h, const float* x, const int64_t stride[3], int32_t B, int32_t T, float* emb, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!h->have_weights) fail(AVC_ERR_STATE, "weights not loaded");
    if (!x || !emb || B <= 0 || T <= 0) fail(AVC_ERR_INVALID, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    Plan plan(&h->pool, st);           // zero fills / uploads ordered on the caller's stream (it may be non-blocking)
    Emitter S{h, &plan.setup, &plan.mem};
    EncActs A = alloc_encoder(plan.mem, h->se, B, T, false, false);
    emit_layout_in(S, x, stride, A.input(h->se), B, h->desc.speaker.c_in);
    emit_bank_and_inconv(S, h->se, A, false);
    emit_encoder_blocks_fwd(S, h->se, A, false);
    TailArgs t = tail_args(h->se, A);
    t.mode = TAIL_FWD; t.emb = emb;
    emit_tail(S, t, B);
    run_list(plan.setup, st);
    h->launches += (long long)plan.setup.size();
    CK(cudaStreamSynchronize(st));
  });
}

int avc_inference(avc_handle* h, const float* src, const int64_t src_stride[3], int32_t T_src, const float* tgt,
                  const int64_t tgt_stride[3], int32_t T_tgt, int32_t B, float* out, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!h->have_weights) fail(AVC_ERR_STATE, "weights not loaded");
    if (!src || !tgt || !out || B <= 0 || T_src <= 0 || T_tgt <= 0) fail(AVC_ERR_INVALID, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    Plan plan(&h->pool, st);
    Emitter S{h, &plan.setup, &plan.mem};
    const int C = h->desc.speaker.c_in, L = content_frames(h, T_src), T_dec = decoder_frames(h, T_src);
    EncActs ce = alloc_encoder(plan.mem, h->ce, B, T_src, false, true);
    EncActs se = alloc_encoder(plan.mem, h->se, B, T_tgt, false, false);
    DecActs dec = alloc_decoder(plan.mem, h->dec, B, L, false);
    float* dout = plan.mem.f((size_t)B * T_dec * C);
    emit_layout_in(S, src, src_stride, ce.input(h->ce), B, C);
    emit_bank_and_inconv(S, h->ce, ce, true);
    emit_encoder_blocks_fwd(S, h->ce, ce, true);
    const int nb = h->ce.d.n_conv_blocks;
    ConvArgs am = fwd_conv_args(h->ce.mean_layer, tens(ce.hout[nb - 1], L, h->ce.d.c_h), tens(dec.z, L, h->ce.d.c_out), B, false, 0.f);
    S.conv(am, &h->ce.mean_layer);
    emit_decoder_const(S, h->dec, dec);
    emit_layout_in(S, tgt, tgt_stride, se.input(h->se), B, C);
    emit_bank_and_inconv(S, h->se, se, false);
    emit_encoder_blocks_fwd(S, h->se, se, false);
    TailArgs t = tail_args(h->se, se);
    t.mode = TAIL_FWD;
    emit_tail(S, t, B);
    emit_decoder_fwd(S, h->dec, dec, se.emb, tens(dout, T_dec, C));
    const int64_t cs[3] = {(int64_t)C * T_dec, (int64_t)T_dec, 1};
    emit_layout_out(S, tens(dout, T_dec, C), out, cs, B, C);
    run_list(plan.setup, st);
    h->launches += (long long)plan.setup.size();
    CK(cudaStreamSynchronize(st));
  });
}

// ---- unit-test entry points ---------------------------------------------------------------------------
static ConvW pack_adhoc(avc_handle* h, Arena& tmp, const float* w_dev, const float* bias_dev, int c_in, int c_out, int k, int stride) {
  std::vector<float> w((size_t)c_out * c_in * k), b(c_out, 0.f);
  CK(cudaMemcpy(w.data(), w_dev, w.size() * sizeof(float), cudaMemcpyDeviceToHost));
  if (bias_dev) CK(cudaMemcpy(b.data(), bias_dev, b.size() * sizeof(float), cudaMemcpyDeviceToHost));
  ConvW c;
  c.c_in = c_in; c.c_out = c_out; c.k = k; c.stride = stride;
  std::vector<float> f((size_t)k * c_in * c_out), r((size_t)k * c_out * c_in);
  for (int n = 0; n < c_out; ++n)
    for (int ci = 0; ci < c_in; ++ci)
      for (int j = 0; j < k; ++j) {
        const float v = w[((size_t)n * c_in + ci) * k + j];
        f[((size_t)j * c_in + ci) * c_out + n] = v;
        r[((size_t)(k - 1 - j) * c_out + n) * c_in + ci] = v;
      }
  c.fwd = tmp.upload(f); c.bwd = tmp.upload(r); c.bias = tmp.upload(b);
  tc_pack_both(tmp, c, f, r);
  (void)h;
  return c;
}

static void check_conv_dims(int B, int T, int c_in, int c_out, int k, int stride) {
  if (B <= 0 || T <= 0 || c_in <= 0 || c_out <= 0 || c_in % 4 || c_out % 4 || k < 1 || k > kMaxTaps || stride < 1 || stride > 4)
    fail(AVC_ERR_INVALID, "conv1d: need channels %% 4 == 0, 1 <= k <= %d, 1 <= stride <= 4", kMaxTaps);
  if (T <= k / 2) fail(AVC_ERR_INVALID, "conv1d: T=%d too short for reflect pad %d", T, k / 2);
}

int avc_conv1d_fwd(avc_handle* h, const float* x, const float* w, const float* bias, float* y, int32_t B, int32_t T,
                   int32_t c_in, int32_t c_out, int32_t k, int32_t stride, int32_t impl, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    check_conv_dims(B, T, c_in, c_out, k, stride);
    Arena tmp(nullptr, (cudaStream_t)stream);
    ConvW c = pack_adhoc(h, tmp, w, bias, c_in, c_out, k, stride);
    const int To = cdiv(T, stride);
    ConvArgs a = fwd_conv_args(c, tens(const_cast<float*>(x), T, c_in), tens(y, To, c_out), B, false, 0.f);
    const int save = h->conv_impl;
    h->conv_impl = impl;
    std::vector<Launch> v;
    try {
      Emitter E{h, &v, &tmp};
      E.conv(a, &c);
      run_list(v, (cudaStream_t)stream);
    } catch (...) { h->conv_impl = save; cudaDeviceSynchronize(); throw; }
    h->conv_impl = save;
    h->launches += (long long)v.size();
    CK(cudaStreamSynchronize((cudaStream_t)stream));
  });
}

int avc_conv1d_dgrad(avc_handle* h, const float* dy, const float* w, float* dx, int32_t B, int32_t T, int32_t c_in,
                     int32_t c_out, int32_t k, int32_t stride, int32_t impl, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    check_conv_dims(B, T, c_in, c_out, k, stride);
    Arena tmp(nullptr, (cudaStream_t)stream);
    ConvW c = pack_adhoc(h, tmp, w, nullptr, c_in, c_out, k, stride);
    const int To = cdiv(T, stride);
    ConvArgs a = bwd_conv_args(c, tens(const_cast<float*>(dy), To, c_out), tens(dx, T, c_in), B, 0.f);
    const int save = h->conv_impl;
    h->conv_impl = impl;
    std::vector<Launch> v;
    try {
      Emitter E{h, &v, &tmp};
      E.conv(a, &c);
      run_list(v, (cudaStream_t)stream);
    } catch (...) { h->conv_impl = save; cudaDeviceSynchronize(); throw; }
    h->conv_impl = save;
    h->launches += (long long)v.size();
    CK(cudaStreamSynchronize((cudaStream_t)stream));
  });
}

// dW[co][ci][j] = sum over splits (fp64, in order) of partial[s][j][ci][co]   (tensor-core path: c_in rows, c_out contiguous)
__global__ void wt_final_1d_kernel(const float* __restrict__ partial, int splits, int k, int c_in, int c_out, float* __restrict__ dw) {
  const long long n = (long long)k * c_in * c_out;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int q = 0; q < splits; ++q) s += (double)partial[(long long)q * n + i];
    const int co = (int)(i % c_out);
    const long long t = i / c_out;
    const int ci = (int)(t % c_in), j = (int)(t / c_in);
    dw[((long long)co * c_in + ci) * k + j] = (float)s;
  }
}

int avc_conv1d_wgrad_ex(avc_handle* h, const float* x, const float* dy, float* dw, float* dbias, int32_t B, int32_t T,
                        int32_t c_in, int32_t c_out, int32_t k, int32_t stride, int32_t impl, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    check_conv_dims(B, T, c_in, c_out, k, stride);
    if (!x || !dy || !dw) fail(AVC_ERR_INVALID, "conv1d_wgrad: null tensor");
    if (impl < 0 || impl > 2) fail(AVC_ERR_INVALID, "conv1d_wgrad: impl %d (0 auto, 1 fp32 CUDA cores, 2 tcgen05)", impl);
    const int To = cdiv(T, stride);
    const long long rows = (long long)B * To;
    cudaStream_t st = (cudaStream_t)stream;
    Arena tmp(&h->pool, st);   // partial tiles / operand planes: slabs recycled through the handle's pool (no cudaMalloc per call)
    const bool tc = impl == 2 || (impl == 0 && rows >= h->tc_min_rows && c_in % 4 == 0 && c_out % 4 == 0 && k <= kWtMaxTaps);
    if (tc) {
      if (c_in % 4 || c_out % 4 || k > kWtMaxTaps) fail(AVC_ERR_INVALID, "conv1d_wgrad: the tensor-core kernel needs channel counts that are multiples of 4 and k <= %d", kWtMaxTaps);
      // operand planes: x reflect-padded (models.py:23-28), both operands split hi / lo for 3xTF32
      const int pl = k / 2, pr = k / 2 - (k % 2 == 0 ? 1 : 0), Tp = T + pl + pr;
      float* xh = tmp.f((size_t)B * Tp * c_in); float* xl = tmp.f((size_t)B * Tp * c_in);
      float* gh = tmp.f((size_t)rows * c_out);  float* gl = tmp.f((size_t)rows * c_out);
      wt_split_pad_kernel<<<ew_grid((long long)B * Tp * c_in / 4, h->sm_count), 256, 0, st>>>(x, xh, xl, B, 1, T, c_in, 0, pl, pr);
      CK(cudaGetLastError());
      wt_split_pad_kernel<<<ew_grid(rows * c_out / 4, h->sm_count), 256, 0, st>>>(dy, gh, gl, B, 1, To, c_out, 0, 0, 0);
      CK(cudaGetLastError());
      WtArgs p{};
      p.a_wmul = stride; p.a_hmul = 1; p.g_wmul = 1; p.g_hmul = 1;
      for (int j = 0; j < k; ++j) { p.a_woff[j] = j; p.a_hoff[j] = 0; p.g_woff[j] = 0; p.g_hoff[j] = 0; }
      p.n_taps = k; p.Ci = c_in; p.Co = c_out; p.Cop = c_out;
      wt_pick_boxes(p, To, 1, B);           // after the taps: the stage geometry depends on which operand moves with the tap
      const int S = wt_splits(p, h->sm_count);
      p.partial = tmp.f((size_t)S * k * c_in * c_out);
      const WtOperand A{xh, xl, c_in, Tp, 1, B, stride, 1}, G{gh, gl, c_out, To, 1, B, 1, 1};
      launch_wgrad_tc(A, G, p, S, st);
      wt_final_1d_kernel<<<ew_grid((long long)k * c_out * c_in, h->sm_count), 256, 0, st>>>(p.partial, S, k, c_in, c_out, dw);
      CK(cudaGetLastError());
      h->launches += 4;
    } else {
      WgradArgs a{};
      a.x = x; a.T = T; a.c_in = c_in; a.dy = dy; a.To = To; a.c_out = c_out;
      a.B = B; a.k = k; a.stride = stride; a.pl = k / 2;
      const int tiles = cdiv(c_out, kWgTile) * cdiv(c_in, kWgTile) * k;
      // enough row splits for ~3 CTAs per SM, at least 64 rows each
      int splits = std::max(1, std::min<int>((int)((rows + 63) / 64), cdiv(3 * h->sm_count, tiles)));
      a.rows_per_split = (int)((rows + splits - 1) / splits);
      a.rows_per_split = cdiv(a.rows_per_split, kWgRows) * kWgRows;
      splits = (int)((rows + a.rows_per_split - 1) / a.rows_per_split);
      a.splits = splits;
      a.partial = tmp.f((size_t)splits * k * c_out * c_in);
      dim3 grid(cdiv(c_out, kWgTile), cdiv(c_in, kWgTile), k * splits);
      conv_wgrad_kernel<<<grid, 256, 0, st>>>(a);
      CK(cudaGetLastError());
      conv_wgrad_final_kernel<<<ew_grid((long long)k * c_out * c_in, h->sm_count), 256, 0, st>>>(a.partial, splits, k, c_out, c_in, dw);
      CK(cudaGetLastError());
      h->launches += 2;
    }
    if (dbias) {
      conv_bgrad_kernel<<<cdiv(c_out, 32), 256, 0, st>>>(dy, rows, c_out, dbias);
      CK(cudaGetLastError());
      h->launches += 1;
    }
    CK(cudaStreamSynchronize(st));
  });
}

int avc_conv1d_wgrad(avc_handle* h, const float* x, const float* dy, float* dw, float* dbias, int32_t B, int32_t T,
                     int32_t c_in, int32_t c_out, int32_t k, int32_t stride, void* stream) {
  return avc_conv1d_wgrad_ex(h, x, dy, dw, dbias, B, T, c_in, c_out, k, stride, 0, stream);
}

int avc_instnorm_adain_act_fwd(avc_handle* h, const float* y, const float* cond, const float* res, int32_t up, float* out,
                               float* stats_out, int32_t B, int32_t T, int32_t C, float neg_slope, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!y || !out || B <= 0 || T <= 0 || C <= 0 || up < 1) fail(AVC_ERR_INVALID, "bad argument");
    if (res && T % up) fail(AVC_ERR_INVALID, "T must be a multiple of up");
    std::vector<Launch> v;
    Arena scratch(nullptr, (cudaStream_t)stream);
    Emitter E{h, &v, &scratch};
    ResArgs r = no_res();
    if (res) r = mk_res(tens(const_cast<float*>(res), T / up, C), up > 1 ? RES_UP : RES_SAME, up);
    emit_norm_fwd(E, y, B, T, C, cond, 2 * C, nullptr, stats_out, out, r, neg_slope);
    run_unit(h, (cudaStream_t)stream, [&] { run_list(v, (cudaStream_t)stream); });
  });
}

int avc_instnorm_adain_act_bwd(avc_handle* h, const float* g, const float* y, const float* stats, const float* cond, float* gy,
                               float* gcond, int32_t B, int32_t T, int32_t C, float neg_slope, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!g || !y || !stats || B <= 0 || T <= 0 || C <= 0 || C % kNormCh) fail(AVC_ERR_INVALID, "bad argument");
    std::vector<Launch> v;
    Arena scratch(nullptr, (cudaStream_t)stream);
    Emitter E{h, &v, &scratch};
    emit_norm_bwd(E, g, y, stats, cond, 2 * C, gy, gcond, 2 * C, B, T, C, neg_slope);
    run_unit(h, (cudaStream_t)stream, [&] { run_list(v, (cudaStream_t)stream); });
  });
}

int avc_adam_tanh_step(avc_handle* h, const float* g_adv, const float* x, float* w, float* m, float* v, float* adv, int64_t n,
                       float eps, int32_t step, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return guarded(h, [&] {
    if (!g_adv || !x || !w || !m || !v || !adv || n <= 0 || n % 4 || step < 1) fail(AVC_ERR_INVALID, "bad argument (n must be a multiple of 4, step >= 1)");
    cudaStream_t st = (cudaStream_t)stream;
    Arena tmp(nullptr, st);
    const double t = step;
    std::vector<float> tab = {(float)(1e-3 / (1.0 - std::pow(0.9, t))), (float)std::sqrt(1.0 - std::pow(0.999, t))};
    UpdateArgs u{};
    u.g_adv = g_adv; u.g_bs = n; u.g_rs = (int)0; u.x = x; u.w = w; u.m = m; u.v = v; u.adv = adv; u.adv_bs = n; u.adv_rs = 0;
    u.B = 1; u.T = 1; u.C = (int)n;   // one row of n channels
    if (n > (1LL << 30)) fail(AVC_ERR_INVALID, "n too large for the unit-test entry point");
    u.eps = eps;
    u.table = reinterpret_cast<float2*>(tmp.upload(tab));
    u.step = tmp.raw<int>(1);
    u.done = nullptr;
    const unsigned g = ew_grid(n / 4, h->sm_count);
    run_unit(h, st, [&] { launch_k(adam_tanh_update_kernel, g, 256, 0, st, u); });
  });
}

#ifdef AVC_SMALL_PROFILE
// debug build only (not part of the C-ABI): copy out and reset the conv_small phase stamps
extern "C" int avc_debug_small_profile(unsigned long long* out, int cap) {
  unsigned n = 0;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(&n, g_small_prof_n, sizeof(n));
  const int m = (int)std::min<unsigned>(std::min<unsigned>(n, 8192u), (unsigned)cap);
  if (m > 0) cudaMemcpyFromSymbol(out, g_small_prof, (size_t)m * 12 * sizeof(unsigned long long));
  n = 0;
  cudaMemcpyToSymbol(g_small_prof_n, &n, sizeof(n));
  return m;
}
#endif
int avc_unit_timing(avc_handle* h, int32_t reps) {
  if (!h || reps < 0 || reps > 1000) return AVC_ERR_INVALID;
  h->unit_reps = reps;
  h->unit_ms = 0.f;
  return AVC_OK;
}
float avc_unit_last_ms(const avc_handle* h) { return h ? h->unit_ms : -1.f; }
int64_t avc_kernel_launches(const avc_handle* h) { return h ? h->launches : -1; }
int32_t avc_launches_per_iter(const avc_handle* h) { return h ? h->launches_per_iter : -1; }

}  // extern "C"
