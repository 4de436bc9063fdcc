// conv_tc.cuh -- tcgen05 / TMEM implicit-GEMM Conv1d for large M (batched attacks), sm_100a only.
//
// Same contraction as conv_simt.cuh (reference pad_layer + nn.Conv1d, models.py:10-30, and its
// autograd w.r.t. the input), on the 5th-generation tensor cores:
//
//   * precision: every value is split a = a_hi + a_lo (a_hi = tf32(a)); per 8 input channels one kind::tf32 MMA
//     D += A_hi*B_hi and ONE kind::f16 BF16 MMA with K = 16 whose rows are [bf16(a_lo) | bf16(a_hi)] x [bf16(b_hi) ;
//     bf16(b_lo)], i.e. D += A_lo*B_hi + A_hi*B_lo, fp32 accumulation in TMEM.  One TF32 pass misses the 1e-3 gradient
//     tolerance by 20x (SURVEY.md §7); this split is ~2^-19 per product and measures 5e-7 per conv.
//   * M axis = "virtual rows": utterances laid end to end with a fixed spacing Pv >= valid rows +
//     taps - 1, so that a conv tap is a pure row shift of ONE shared-memory window even when a
//     128-row tile spans several (short) utterances.  Rows past an utterance's valid range are dead.
//   * A operand: loader warps gather the window from global memory (reflect padding / zero padding
//     and the optional act' mask by index arithmetic), split every value and store the TF32 plane and the
//     bf16-pair plane in the UMMA "interleaved" (no-swizzle, K-major) canonical layout
//     [k/4][row][4 floats]: core matrices of consecutive 8-row groups are contiguous (SBO = 128 B),
//     so tap j is the SAME buffer with the descriptor start address advanced by j*16 bytes.
//   * B operand: weights pre-split and pre-tiled on the host in exactly the shared-memory image of
//     one (K-block, tap) stage, streamed by one elected thread with cp.async.bulk (TMA engine,
//     mbarrier complete_tx) through a ring.
//   * one elected thread issues tcgen05.mma (kind::tf32, M=128, N <= 128); tcgen05.commit frees the
//     ring slots and signals the drain warps.
//   * accumulation is CHUNKED: the tensor core accumulates fp32 with truncation, a bias that grows
//     linearly with the number of MMA steps (measured: -8e-8 relative per K=8 step, 3.3e-6 at K=640).
//     So every 12 k-steps (24 MMAs) the accumulator (a ring of four 128-column TMEM buffers) is handed to eight
//     drain warps, which add it into fp32 registers with round-to-nearest (tcgen05.ld), and finally apply bias /
//     act' mask / activation / residual exactly like the CUDA-core kernel.
//   * the (pass, group, K block, tap, chunk) walk is a host-built table in the kernel parameters (TcStage).
//   * dgrad: the transposed conv is evaluated on the EXTENDED row range [-pl, T+pr); the rows outside
//     [0,T) (gradient of the reflect padding) go to a small side buffer and `tc_fold_kernel` adds them
//     to their mirror rows -- no atomics, fixed order.
//
//   * strided convs: forward = one group per tap residue (parity planes of the input); dgrad = one
//     pass per output residue.  N > 128 (decoder up-convs, in-conv dgrad) = one pass per 128 columns.
#pragma once
#include <cstdint>
#include <vector>

#include "conv_simt.cuh"
#include "host_util.h"
#include "tc_common.cuh"

namespace avc {

constexpr int kTcM = 128;          // rows of one UMMA / one CTA tile
constexpr int kTcRows = 136;       // window rows per A stage (128 + kMaxTaps)
constexpr int kTcKB = 32;          // channels per K block (4 UMMA k-steps of 8)
constexpr int kTcAStages = 2;
constexpr int kTcBStages = 3;
constexpr int kTcNMax = 128;       // columns of one pass
constexpr int kTcThreads = 448;    // warp 0: TMEM + weight producer, 1: MMA issuer, 2-5: loaders, 6-13: drain + epilogue
constexpr int kTcAPlane = (kTcKB / 4) * kTcRows * 4;   // floats of one hi (or lo) plane of an A stage
constexpr int kTcChunkSteps = 12;  // default MMA k-steps (2 MMAs each) accumulated in TMEM before the drain warps take over: 24 accumulate operations, see DESIGN.md
constexpr int kTcAccBufs = 4;      // accumulator ring in TMEM (4 x 128 columns = all 512): hides the drain hand-off latency
constexpr int kTcMaxChunks = 12;   // N chunks of one packed conv (1104 = 8 x 128 + 80)
constexpr int kTcMaxPass = 12;
#ifndef AVC_TC_PF_DIST
#define AVC_TC_PF_DIST 3
#endif
constexpr int kTcPfDist = AVC_TC_PF_DIST;   // K blocks of window rows prefetched into L2 ahead of the loaders' register fetch

struct TcPack {                    // weights of ONE conv direction / tap subset, device memory
  bool ok = false;
  int k = 0, kc = 0, n = 0, n_chunks = 0;
  float* blocks[kTcMaxChunks] = {};   // per N chunk: [kb][tap][plane hi|lo][k/4][cn][4]
  int cn[kTcMaxChunks] = {};
};

struct TcGroup {
  const float* Wp;                 // packed blocks of this group (for this pass's N chunk)
  int a_ch_off, kc, n_taps;
  int sg, off0;                    // input position of window row u:  sg*u + off0
};

struct TcPass {
  int g_begin, g_end;              // groups accumulated by this pass
  int N, ch_off;                   // columns of this pass and where they go in the output row
  int so, oo;                      // output index of virtual row u:  so*u + oo
  int s_begin, s_end;              // its weight stages in TcArgs::st (tc_build_stages)
  int n_chunks;                    // accumulator hand-offs to the drain warps
};

// One weight stage = one (K block, tap) of one group.  The table is worked out on the host and travels in the
// kernel parameters (constant bank: the producer and the MMA issuer read it with uniform loads), so no role
// re-derives the (group, K block, tap, chunk) walk on the device.
constexpr int kTcMaxStages = 192;
enum : unsigned { kTcKbFirst = 1, kTcKbLast = 2, kTcChunkFirst = 4, kTcChunkLast = 8 };
struct TcStage {
  uint32_t w_off;                  // float offset of its hi|lo weight block from the group's Wp
  uint8_t gi, tap, nks, flags;     // group, window shift (rows), MMA k-steps, kTc* flags
};

struct TcArgs {
  const float* A; long long a_bs; int a_rs; int T_a;
  const float* Mk; long long m_bs; int m_rs; float slope;
  int bwd;               // 0: reflect gather (forward), 1: zero-padded gather (dgrad)
  int Pv;                // virtual rows per utterance
  int T_y;               // main output rows per utterance
  int halo_l, halo_r;    // dgrad: rows kept on each side for the reflect-pad fold
  int B; long long Mv;   // B * Pv
  int side_n;            // columns of one side-buffer row (the whole output width)
  float* Y; long long y_bs; int y_rs;
  float* Y2; long long y2_bs; int y2_rs;
  const float* bias; int act;
  const float* Om; long long om_bs; int om_rs;
  ResArgs res;
  float* side;           // [B][halo_l + halo_r][side_n]
  int n_pass;
  int terms;             // >= 2: TF32 hi*hi + BF16 correction MMA (product), 1: single TF32 pass (measurement only)
  int chunk_steps;       // MMA k-steps accumulated in TMEM before the drain warps take the partial sum (env AVC_TC_CHUNK)
  int dbg;               // bottleneck probes (results are garbage): 1 no weight copies, 2 no window gather, 4 no MMA
  TcPass pass[kTcMaxPass];
  TcGroup g[kTcMaxPass];
  TcStage st[kTcMaxStages];
  // Ragged batches (kernels instantiated with VL = true): per-utterance valid rows of the input (T_a), the output (T_y) and
  // the skip tensor (res.T_r), device int32 [B].  The scalar fields then hold the padded maxima.  Appended last so that the
  // equal-length kernels keep their parameter offsets.
  const int* lens_a; const int* lens_y; const int* lens_r;
};

// ---- host: weight packing ----------------------------------------------------------------------
inline float tf32_hi_host(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  u = (u + 0x1000u) & 0xffffe000u;   // round to 10 mantissa bits (ties away), same as the device split
  float r;
  memcpy(&r, &u, 4);
  return r;
}

inline uint16_t bf16_rn_host(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  u += 0x7fffu + ((u >> 16) & 1u);   // round to nearest even on the top 16 bits (finite inputs)
  return (uint16_t)(u >> 16);
}

// img: [k_img][kc][n] (n contiguous) -- the forward or dgrad image pack_conv builds for the CUDA-core
// path; taps: which taps of the image, in window order, this pack contracts.
inline void tc_pack_taps(Arena& mem, TcPack& p, const std::vector<float>& img, int kc, int n, const std::vector<int>& taps) {
  const int k = (int)taps.size();
  p.ok = false; p.k = k; p.kc = kc; p.n = n; p.n_chunks = 0;
  if (kc % 8 || n % 8 || k < 1 || k > kMaxTaps) return;
  const int nch = (n + kTcNMax - 1) / kTcNMax;
  if (nch > kTcMaxChunks) return;
  for (int ch = 0; ch < nch; ++ch) {
    const int cn = std::min(kTcNMax, n - ch * kTcNMax);
    if (cn != 128 && cn != 80) return;   // drain warps are instantiated for 64 / 40 columns per thread
  }
  const int nkb = (kc + kTcKB - 1) / kTcKB;
  for (int ch = 0; ch < nch; ++ch) {
    const int n0 = ch * kTcNMax, cn = std::min(kTcNMax, n - n0);
    // two images back to back: [0] whole stages for the single-CTA kernel, [1] the same stages split into column halves
    // for the CTA-pair kernel ([half][plane][k/4][cn/2][16 B], each CTA streams its half)
    const size_t img_floats = (size_t)2 * k * kc * cn;
    std::vector<float> out(2 * img_floats);
    uint16_t* out16 = reinterpret_cast<uint16_t*>(out.data());
    size_t o = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      const int kb0 = kb * kTcKB, kbs = std::min(kTcKB, kc - kb0);
      for (int t = 0; t < k; ++t) {
        auto wv = [&](int c, int nn) { return img[((size_t)taps[t] * kc + kb0 + c) * n + n0 + nn]; };
        // plane 0: TF32 hi parts, [k/4][n][4 floats]
        for (int c = 0; c < kbs / 4; ++c)
          for (int nn = 0; nn < cn; ++nn)
            for (int e = 0; e < 4; ++e) {
              const float hi = tf32_hi_host(wv(4 * c + e, nn));
              out[o + ((size_t)c * cn + nn) * 4 + e] = hi;
              const int h = nn / (cn / 2), nh = nn % (cn / 2);
              out[img_floats + o + (size_t)h * kbs * cn + ((size_t)c * (cn / 2) + nh) * 4 + e] = hi;
            }
        // plane 1: per MMA k-step of 8 channels two 16-byte K chunks per column: bf16(hi[0..8)), bf16(lo[0..8))
        for (int ks = 0; ks < kbs / 8; ++ks)
          for (int j = 0; j < 2; ++j)
            for (int nn = 0; nn < cn; ++nn)
              for (int e = 0; e < 8; ++e) {
                const float v = wv(8 * ks + e, nn);
                const float hi = tf32_hi_host(v);
                const uint16_t q = bf16_rn_host(j == 0 ? hi : v - hi);
                out16[2 * (o + (size_t)kbs * cn) + ((size_t)(2 * ks + j) * cn + nn) * 8 + e] = q;
                const int h = nn / (cn / 2), nh = nn % (cn / 2);
                out16[2 * (img_floats + o + (size_t)h * kbs * cn + (size_t)kbs * cn / 2) + ((size_t)(2 * ks + j) * (cn / 2) + nh) * 8 + e] = q;
              }
        o += (size_t)2 * kbs * cn;
      }
    }
    p.blocks[ch] = mem.upload(out);
    p.cn[ch] = cn;
  }
  p.n_chunks = nch;
  p.ok = true;
}

// device helpers (mbarrier, tcgen05, TMEM): tc_common.cuh

constexpr int kTcBarSlots = 38;    // 8-byte slots of the barrier block (36 barriers + the TMEM address)
constexpr int kTcScrPitch = 36;    // floats per row of a drain warp's transpose slab (32 + 4: conflict-free float4 rows)

// ---- epilogue ------------------------------------------------------------------------------------
// Each drain lane owns one accumulator ROW; rows are 512 B apart in memory, so the tile is transposed
// through a per-warp shared-memory slab and written with lanes along the channel axis.  Everything that
// depends on the row (utterance, output row, which rows of the skip tensor it reads, their weight) is
// worked out ONCE by the lane that owns the row and handed to the storing lanes with shuffles, and the
// row loop is a real loop: the whole kernel has to stay a few tens of KB of code (the first version
// unrolled 16 row groups x 5 skip modes per tile, 370 KB of SASS, and the drain warps spent 10-20k clk
// per tile fetching instructions).
struct TcRow {
  int kind;      // 0 dead, 1 main row, 2 dgrad halo row
  int b, o;      // utterance, output row (kind 2: row of the side buffer)
  int t0, t1;    // rows of the skip tensor (t1 < 0: one row only)
  float rs;      // skip value = (R[t0] + R[t1]) * rs
};

__device__ __forceinline__ TcRow tc_row_info(const TcArgs& p, const TcPass& ps, long long u) {
  TcRow r;
  r.b = (int)(u / p.Pv);
  r.o = ps.so * (int)(u - (long long)r.b * p.Pv) + ps.oo;
  r.kind = 0; r.t0 = 0; r.t1 = -1; r.rs = 1.f;
  if (r.b < p.B && !(p.dbg & 8)) {
    if (r.o >= 0 && r.o < p.T_y) r.kind = 1;
    else if (p.side && ((r.o < 0 && r.o >= -p.halo_l) || (r.o >= p.T_y && r.o < p.T_y + p.halo_r))) {
      r.kind = 2;
      r.o = r.o < 0 ? r.o + p.halo_l : p.halo_l + (r.o - p.T_y);
    }
  }
  if (r.kind == 1) {
    const int rf = p.res.rf, t = r.o;
    switch (p.res.mode) {   // res_load4 (common.cuh) with the loads separated from the index arithmetic; rf <= 2 (tc_supported)
      case RES_SAME: r.t0 = t; break;
      case RES_POOL: { const int lo = t * rf, n = min(rf, p.res.T_r - lo); r.t0 = lo; r.t1 = n > 1 ? lo + 1 : -1; r.rs = 1.f / (float)n; break; }
      case RES_POOL_BWD: { const int q = rf > 1 ? t >> 1 : t; r.t0 = q; r.rs = 1.f / (float)min(rf, p.T_y - q * rf); break; }
      case RES_UP: r.t0 = rf > 1 ? t >> 1 : t; break;
      case RES_UP_BWD: r.t0 = t * rf; r.t1 = rf > 1 ? t * rf + 1 : -1; break;
      default: break;
    }
  }
  return r;
}

// Ragged batches: the same with every length read from the utterance's entry of the tables (b is checked against B first:
// the last tile runs past the batch).  A separate function rather than a branch inside tc_row_info so that the
// equal-length kernels keep their instruction streams.
__device__ __forceinline__ TcRow tc_row_info_vl(const TcArgs& p, const TcPass& ps, long long u) {
  TcRow r;
  r.b = (int)(u / p.Pv);
  r.o = ps.so * (int)(u - (long long)r.b * p.Pv) + ps.oo;
  r.kind = 0; r.t0 = 0; r.t1 = -1; r.rs = 1.f;
  int T_y = 0;
  if (r.b < p.B && !(p.dbg & 8)) {
    T_y = p.lens_y[r.b];
    if (r.o >= 0 && r.o < T_y) r.kind = 1;
    else if (p.side && ((r.o < 0 && r.o >= -p.halo_l) || (r.o >= T_y && r.o < T_y + p.halo_r))) {
      r.kind = 2;
      r.o = r.o < 0 ? r.o + p.halo_l : p.halo_l + (r.o - T_y);
    }
  }
  if (r.kind == 1) {
    const int rf = p.res.rf, t = r.o;
    switch (p.res.mode) {   // the speaker encoder's skip modes
      case RES_SAME: r.t0 = t; break;
      case RES_POOL: { const int lo = t * rf, n = min(rf, p.lens_r[r.b] - lo); r.t0 = lo; r.t1 = n > 1 ? lo + 1 : -1; r.rs = 1.f / (float)n; break; }
      case RES_POOL_BWD: { const int q = rf > 1 ? t >> 1 : t; r.t0 = q; r.rs = 1.f / (float)min(rf, T_y - q * rf); break; }
      default: break;
    }
  }
  return r;
}

template <bool VL>
__device__ __forceinline__ TcRow tc_row(const TcArgs& p, const TcPass& ps, long long u) {
  if constexpr (VL) return tc_row_info_vl(p, ps, u);
  else return tc_row_info(p, ps, u);
}

// Ragged batches: the row of utterance b's input that window position pos reads (reflect padding around the utterance's
// own length in the forward, zeros outside it in the dgrad), -1 for zeros
__device__ __forceinline__ int tc_src_row_vl(const TcArgs& p, int b, int pos) {
  if (b >= p.B) return -1;
  const int T_a = p.lens_a[b];
  int rr = pos;
  if (!p.bwd) {
    rr = rr < 0 ? -rr : rr;
    if (rr >= T_a) rr = 2 * (T_a - 1) - rr;
  }
  return rr >= 0 && rr < T_a ? rr : -1;
}

#ifndef AVC_TC_EPI_BATCH
#define AVC_TC_EPI_BATCH 4
#endif
// Columns [chb, chb+SW) of the 32 rows a drain warp owns, slab -> global.  SW/4 lanes per row, so a warp
// instruction covers 32/(SW/4) rows with contiguous SW*4-byte segments.  Rows go in batches of NB: all the
// global loads of a batch (act' mask, skip rows) are in flight before the first one is consumed.
// ncol: valid columns of the slab (a pass of N = 80 fills 64 + 16 of the two 64-column halves).
__device__ __forceinline__ void tc_slab_to_global(const TcArgs& p, const float* scratch, int lane, const TcRow& own, int chb, int ncol) {
  constexpr int SW = 32, LPR = SW / 4, RPI = 32 / LPR, ITS = 32 / RPI;
  constexpr int NB = ITS < AVC_TC_EPI_BATCH ? ITS : AVC_TC_EPI_BATCH;
  const int c4 = lane % LPR, ch = chb + 4 * c4, rsub = lane / LPR;
  const bool col_ok = 4 * c4 < ncol;
  const float4 bias = (p.bias && col_ok) ? ld4(p.bias + ch) : f4zero();
  const bool has_res = p.res.mode != RES_NONE;
#pragma unroll 1
  for (int it0 = 0; it0 < ITS; it0 += NB) {
    int kq[NB], bq[NB], oq[NB];
    float4 om[NB], ra[NB], rb[NB];
    float rsc[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int r = (it0 + j) * RPI + rsub;
      kq[j] = __shfl_sync(0xffffffffu, own.kind, r);
      if (!col_ok) kq[j] = 0;
      bq[j] = __shfl_sync(0xffffffffu, own.b, r);
      oq[j] = __shfl_sync(0xffffffffu, own.o, r);
      om[j] = f4zero(); ra[j] = f4zero(); rb[j] = f4zero(); rsc[j] = 1.f;
      if (p.Om && kq[j] == 1) om[j] = ld4(p.Om + (long long)bq[j] * p.om_bs + (long long)oq[j] * p.om_rs + ch);
      if (has_res) {
        const int t0 = __shfl_sync(0xffffffffu, own.t0, r), t1 = __shfl_sync(0xffffffffu, own.t1, r);
        rsc[j] = __shfl_sync(0xffffffffu, own.rs, r);
        if (kq[j] == 1) {
          const float* rbase = p.res.R + (long long)bq[j] * p.res.bs + ch;
          ra[j] = ld4(rbase + (long long)t0 * p.res.rs);
          if (t1 >= 0) rb[j] = ld4(rbase + (long long)t1 * p.res.rs);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      if (kq[j] == 0) continue;
      const int r = (it0 + j) * RPI + rsub;
      float4 x = ld4(scratch + r * kTcScrPitch + 4 * c4);
      if (kq[j] == 1) {
        if (p.bias) x = f4add(x, bias);
        if (p.Om) x = dact4mul(x, om[j], p.slope);
        if (p.act) x = act4(x, p.slope);
        if (p.Y2) st4(p.Y2 + (long long)bq[j] * p.y2_bs + (long long)oq[j] * p.y2_rs + ch, x);
        if (has_res) x = f4add(x, f4scale(f4add(ra[j], rb[j]), rsc[j]));
        st4(p.Y + (long long)bq[j] * p.y_bs + (long long)oq[j] * p.y_rs + ch, x);
      } else {
        st4(p.side + ((long long)bq[j] * (p.halo_l + p.halo_r) + oq[j]) * p.side_n + ch, x);
      }
    }
  }
}

// registers -> slab: lane's row, columns [C0, C0+32)
template <int NH, int C0>
__device__ __forceinline__ void tc_acc_to_slab(const float (&acc)[NH], float* scratch, int lane) {
#pragma unroll
  for (int q = 0; q < 8; ++q)
    st4(scratch + lane * kTcScrPitch + 4 * q, make_float4(acc[C0 + 4 * q], acc[C0 + 4 * q + 1], acc[C0 + 4 * q + 2], acc[C0 + 4 * q + 3]));
}

constexpr int kTcNH = 64;   // accumulator columns per drain thread (half of a 128-column pass; N = 80: 64 + 16)
#ifndef AVC_TC_DIRECT_EPI
#define AVC_TC_DIRECT_EPI 0
#endif
constexpr bool kTcDirectEpi = AVC_TC_DIRECT_EPI != 0;
// Direct epilogue: every drain lane writes the 64 columns of ITS row straight from its accumulator registers, 16 bytes
// per store.  A warp store touches 32 rows x 16 B (two stores fill a 32-byte sector), which the memory system takes
// at 32 lines per instruction -- but it is ~250 instructions per tile and thread where the transposing version
// (per-warp shared-memory slab, shuffled row descriptors, 64-bit address arithmetic per row group) needs ~1900, and
// the drain warps' instruction stream, not the memory system, is what made the epilogue (~10k clk per tile) longer
// than the accumulator ring lets the MMA issuer run ahead.
template <int NQ>   // float4 columns per batch: the batch's mask / skip loads are in flight before the first is consumed
__device__ __forceinline__ void tc_store_row_batches(const TcArgs& p, const float (&acc)[kTcNH], float* yp, float* y2p,
                                                     const float* g0p, const float* g1p, float rs, int chb, int ncol) {
  const bool has_om = p.Om != nullptr, has_res = p.res.mode != RES_NONE;
#pragma unroll
  for (int q0 = 0; q0 < kTcNH / 4; q0 += NQ) {
    if (4 * q0 < ncol) {
      float4 ga[NQ], gb[NQ];
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        if (g0p) ga[i] = ld4(g0p + 4 * (q0 + i));
        if (g1p) gb[i] = ld4(g1p + 4 * (q0 + i));
      }
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        const int c = 4 * (q0 + i);
        if (c < ncol) {
          float4 x = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
          if (p.bias) x = f4add(x, ld4(p.bias + chb + c));          // same address in every lane: one transaction
          if (has_om) x = dact4mul(x, ga[i], p.slope);
          if (p.act) x = act4(x, p.slope);
          if (y2p) st4(y2p + c, x);
          if (has_res) x = f4add(x, f4scale(g1p ? f4add(ga[i], gb[i]) : ga[i], rs));
          st4(yp + c, x);
        }
      }
    }
  }
}

__device__ __forceinline__ void tc_store_row_direct(const TcArgs& p, const float (&acc)[kTcNH], const TcRow& own, int chb, int ncol) {
  if (own.kind == 0) return;
  if (own.kind == 2) {       // dgrad halo row -> side buffer (own.o is its row there)
    float* sp = p.side + ((long long)own.b * (p.halo_l + p.halo_r) + own.o) * p.side_n + chb;
#pragma unroll
    for (int c = 0; c < kTcNH; c += 4)
      if (c < ncol) st4(sp + c, make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]));
    return;
  }
  float* yp = p.Y + (long long)own.b * p.y_bs + (long long)own.o * p.y_rs + chb;
  float* y2p = p.Y2 ? p.Y2 + (long long)own.b * p.y2_bs + (long long)own.o * p.y2_rs + chb : nullptr;
  if (p.Om) {
    tc_store_row_batches<4>(p, acc, yp, y2p, p.Om + (long long)own.b * p.om_bs + (long long)own.o * p.om_rs + chb, nullptr, 1.f, chb, ncol);
  } else if (p.res.mode != RES_NONE) {
    const float* rb = p.res.R + (long long)own.b * p.res.bs + chb;
    tc_store_row_batches<2>(p, acc, yp, y2p, rb + (long long)own.t0 * p.res.rs, own.t1 >= 0 ? rb + (long long)own.t1 * p.res.rs : nullptr,
                            own.rs, chb, ncol);
  } else {
    tc_store_row_batches<4>(p, acc, yp, y2p, nullptr, nullptr, 1.f, chb, ncol);
  }
}

struct TcDrainProf { long long wait, ld, epi; };
#ifdef AVC_TC_PROFILE
#define TCD(x) x
#else
#define TCD(x)
#endif
template <bool VL>
__device__ __forceinline__ void tc_drain_and_store(const TcArgs& p, const TcPass& ps, uint32_t tmem_base, uint32_t acc_full0,
                                                   uint32_t acc_empty0, long long v0, int warp, int lane, int& chunk, float* scratch,
                                                   TcDrainProf& dp, int leader_rank = -1) {   // >= 0: acc_empty lives in that CTA of the pair
  TCD(long long dq;)
  constexpr int NH = kTcNH;
  const int quad = warp & 3;                    // TMEM lanes this warp may read: [32*quad, 32*quad+32)
  const int half = (warp - 6) >> 2;             // which half of the columns
  const int ncol = min(NH, ps.N - half * NH);   // valid columns of this half
  float acc[NH];
#pragma unroll
  for (int i = 0; i < NH; ++i) acc[i] = 0.f;
  const TcRow own = tc_row<VL>(p, ps, v0 + quad * 32 + lane);   // worked out while the first chunk's MMAs run
  if (own.kind == 1 && kTcPfDist > 0) {   // the epilogue's operands for this lane's row: into L2 now, read ~20k clk later
    const int c0 = ps.ch_off + half * NH;
    if (p.Om) {
      const float* q = p.Om + (long long)own.b * p.om_bs + (long long)own.o * p.om_rs + c0;
      prefetch_l2(q); if (ncol > 32) prefetch_l2(q + 32);
    }
    if (p.res.mode != RES_NONE) {
      const float* q = p.res.R + (long long)own.b * p.res.bs + c0;
      prefetch_l2(q + (long long)own.t0 * p.res.rs); if (ncol > 32) prefetch_l2(q + (long long)own.t0 * p.res.rs + 32);
      if (own.t1 >= 0) { prefetch_l2(q + (long long)own.t1 * p.res.rs); if (ncol > 32) prefetch_l2(q + (long long)own.t1 * p.res.rs + 32); }
    }
  }
#pragma unroll 1
  for (int c = 0; c < ps.n_chunks; ++c) {
    const int buf = chunk % kTcAccBufs;
    TCD(dq = clock64();)
    mbar_wait(acc_full0 + 8 * buf, (chunk / kTcAccBufs) & 1);
    TCD(dp.wait += clock64() - dq; dq = clock64();)
    tc_fence_after();
    const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * kTcNMax + half * NH);
    if (!(p.dbg & 16)) {
      // loads are issued in batches of 32 columns before one wait: the TMEM read latency is paid per batch
#pragma unroll
      for (int c0 = 0; c0 < NH; c0 += 32) {
        if (c0 < ncol) {
          uint32_t r0[16], r1[16];
          tmem_ld16(t0 + c0, r0);
          tmem_ld16(t0 + c0 + 16, r1);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) { acc[c0 + i] += __uint_as_float(r0[i]); acc[c0 + 16 + i] += __uint_as_float(r1[i]); }   // round-to-nearest fp32 adds
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) { if (leader_rank >= 0) mbar_arrive_cta(acc_empty0 + 8 * buf, (uint32_t)leader_rank); else mbar_arrive(acc_empty0 + 8 * buf); }
    TCD(dp.ld += clock64() - dq;)
    ++chunk;
  }
  TCD(dq = clock64();)
  // ---- epilogue: bias / mask / act / residual -> global (overlaps the next tile's MMAs) ----
  const int chb = ps.ch_off + half * NH;
  if (kTcDirectEpi) tc_store_row_direct(p, acc, own, chb, ncol);
  else {
    tc_acc_to_slab<NH, 0>(acc, scratch, lane);
    __syncwarp();
    tc_slab_to_global(p, scratch, lane, own, chb, ncol);
    if (ncol > 32) {
      __syncwarp();
      tc_acc_to_slab<NH, 32>(acc, scratch, lane);
      __syncwarp();
      tc_slab_to_global(p, scratch, lane, own, chb + 32, ncol - 32);
    }
    __syncwarp();
  }
  TCD(dp.epi += clock64() - dq;)
}

// Persistent: gridDim.x CTAs (one per SM) walk the work items (M tile, pass) round-robin; barrier phases,
// ring positions and the accumulator ping-pong run on across items, so the drain warps' epilogue of one
// item overlaps the MMAs of the next.
//
// PAIR = true: the kernel is launched as clusters of two CTAs (one TPC).  The two CTAs work on M tiles 2i and 2i+1 of
// the same pass; the even CTA (the leader) issues cta_group::2 MMAs with M = 256 for both.  Each CTA gathers its own
// window, keeps its own accumulators and runs its own epilogue, but holds only HALF of every weight stage (N/2
// columns): the tensor cores of both SMs read it across the pair.  Per MMA a CTA's shared memory delivers 4 KB of A
// and 2 KB of B instead of 4 + 4, and the bulk copies write 16 KB per stage instead of 32 -- shared-memory bandwidth
// is what bounds the single-CTA kernel (DESIGN.md).  Cross-CTA protocol: the peer's loader and drain warps arrive on
// the LEADER's a_full / acc_empty barriers; the peer's warp 1 forwards "my weight half has landed" to the leader's
// b_fwd barrier; the leader's commits are multicast to the same barrier in both CTAs.
//
// VL = true: ragged batch, lengths from p.lens_* (see TcArgs).
template <bool PAIR, bool VL = false>
__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_kernel_t(const TcArgs p) {
  extern __shared__ __align__(128) unsigned char tc_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int NBS = PAIR ? 2 * kTcBStages : kTcBStages;                            // weight ring depth (half-size stages in a pair)
  constexpr uint32_t b_stage_bytes = 2 * (kTcKB / 4) * kTcNMax * 16 / (PAIR ? 2 : 1);   // both planes of a full weight stage (pair: of its half)
  float* As = reinterpret_cast<float*>(tc_smem);                                     // [kTcAStages][2][kTcAPlane]
  unsigned char* Bs = tc_smem + (size_t)kTcAStages * 2 * kTcAPlane * 4;              // [NBS][b_stage_bytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(Bs + (size_t)kTcBStages * 2 * (kTcKB / 4) * kTcNMax * 16);
  // bars: a_full[2] a_empty[2] b_full[8] b_empty[8] b_fwd[8] acc_full[4] acc_empty[4]
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s) { return bar0 + 8 * s; };
  auto a_empty = [&](int s) { return bar0 + 8 * (2 + s); };
  auto b_full = [&](int s) { return bar0 + 8 * (4 + s); };
  auto b_empty = [&](int s) { return bar0 + 8 * (12 + s); };
  auto b_fwd = [&](int s) { return bar0 + 8 * (20 + s); };
  const uint32_t acc_full0 = bar0 + 8 * 28, acc_empty0 = bar0 + 8 * 32;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);
  float* scr_all = reinterpret_cast<float*>(bars + kTcBarSlots);                      // [8 drain warps][32][kTcScrPitch]
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;                               // 0: leader

  if (threadIdx.x == 0) {
    for (int s = 0; s < kTcAStages; ++s) { mbar_init(a_full(s), PAIR ? 8 : 4); mbar_init(a_empty(s), 1); }
    for (int s = 0; s < 8; ++s) { mbar_init(b_full(s), 1); mbar_init(b_empty(s), 1); mbar_init(b_fwd(s), 1); }
    for (int s = 0; s < kTcAccBufs; ++s) { mbar_init(acc_full0 + 8 * s, 1); mbar_init(acc_empty0 + 8 * s, PAIR ? 16 : 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr uint32_t tmem_cols = kTcAccBufs * kTcNMax;     // accumulator ring
  if (PAIR) cluster_sync_all();                            // both CTAs' barriers exist before anyone arrives remotely
  if (warp == 0) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();

  const int n_mt = (int)((p.Mv + kTcM - 1) / kTcM);
  // item w: M tile (pair: tile pair) w / n_pass, pass w % n_pass (passes of a tile share A in L2)
  const int n_work = (PAIR ? (n_mt + 1) / 2 : n_mt) * p.n_pass;
  const int w_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, w_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  auto tile_row0 = [&](int wk) { return (long long)(PAIR ? 2 * (wk / p.n_pass) + (int)rank : wk / p.n_pass) * kTcM; };   // a tile past the end is all dead rows

  if (warp == 0) {
    // ===== weight producer: one elected lane streams the stages of the table with the TMA engine =====
    if (lane == 0) {
      int sb = 0; uint32_t pb = 0;
      for (int wk = w_first; wk < n_work; wk += w_step) {
        const TcPass& ps = p.pass[wk % p.n_pass];
        const uint32_t N = (uint32_t)ps.N;
#pragma unroll 1
        for (int s = ps.s_begin; s < ps.s_end; ++s) {
          const TcStage e = p.st[s];
          const uint32_t bytes = (PAIR ? 32u : 64u) * e.nks * N;      // 2 planes x (8 nks) channels x N (pair: N/2) x 4 bytes
          const TcGroup& G = p.g[e.gi];
          // pair image: after the single-CTA image (2 * taps * channels * N floats), each stage as [half][plane][k/4][N/2][4]
          const float* src = G.Wp + e.w_off + (PAIR ? (size_t)2 * G.n_taps * G.kc * N + rank * (bytes >> 2) : (size_t)0);
          mbar_wait(b_empty(sb), pb ^ 1);
          if (p.dbg & 1) { mbar_arrive(b_full(sb)); }
          else {
            mbar_expect_tx(b_full(sb), bytes);
            bulk_g2s(smem_u32(Bs + (size_t)sb * b_stage_bytes), src, bytes, b_full(sb));
          }
          if (++sb == NBS) { sb = 0; pb ^= 1; }
        }
      }
    }
  } else if (warp == 1 && PAIR && rank != 0) {
    // ===== peer CTA: forward "my half of weight stage s has landed" to the leader's b_fwd barrier =====
    int sb = 0; uint32_t pb = 0;
    for (int wk = w_first; wk < n_work; wk += w_step) {
      const TcPass& ps = p.pass[wk % p.n_pass];
#pragma unroll 1
      for (int s = ps.s_begin; s < ps.s_end; ++s) {
        mbar_wait(b_full(sb), pb);
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(b_fwd(sb), 0);
        if (++sb == NBS) { sb = 0; pb ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp walks the stage table (waits included), one elected lane issues =====
    {
      const bool leader = elect_one();
      int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
      int chunk = 0;
#ifdef AVC_TC_PROFILE
      long long st_a = 0, st_b = 0, st_acc = 0, st_issue = 0, t_begin = clock64(), tq;   // where the issuer waits (build with -DAVC_TC_PROFILE, run with AVC_TC_DBG=32)
#define TCP(x) x
#else
#define TCP(x)
#endif
      const int terms = p.terms;
      const bool no_mma = (p.dbg & 4) != 0;
      const uint32_t a_base = smem_u32(As), b_base = smem_u32(Bs);
      constexpr uint32_t a_lbo = kTcRows * 16;
      constexpr uint64_t a_lo_off = (uint64_t)((kTcAPlane * 4) >> 4), a_ks = (uint64_t)((2 * a_lbo) >> 4);
      for (int wk = w_first; wk < n_work; wk += w_step) {
        const TcPass& ps = p.pass[wk % p.n_pass];
        const uint32_t N = (uint32_t)ps.N;
        constexpr uint32_t m_field = (uint32_t)((PAIR ? 2 * kTcM : kTcM) >> 4) << 24;                                // M = 256 across the pair
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | m_field;   // TF32 x TF32 -> fp32
        const uint32_t idesc16 = (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | m_field;  // BF16 x BF16 -> fp32, K = 16
        const uint32_t b_lbo = (PAIR ? N / 2 : N) * 16;                                                               // this CTA's columns of the stage
        const uint64_t b_ks = (uint64_t)((2 * b_lbo) >> 4);
        uint64_t a_desc0 = 0;
        uint32_t d_tmem = 0, acc = 0;
#pragma unroll 1
        for (int s = ps.s_begin; s < ps.s_end; ++s) {
          const TcStage e = p.st[s];
          if (e.flags & kTcKbFirst) {
            TCP(tq = clock64();)
            mbar_wait(a_full(sa), pa);
            TCP(if (st_issue == 0) t_begin = clock64(); else st_a += clock64() - tq;)   // the first window also waits for the predecessor kernel (PDL)
            a_desc0 = tc_desc(a_base + (uint32_t)sa * (2 * kTcAPlane * 4), a_lbo, 128);
          }
          if (e.flags & kTcChunkFirst) {     // first stage of a chunk: wait for the drain warps to release the buffer
            const int buf = chunk % kTcAccBufs;
            TCP(tq = clock64();)
            mbar_wait(acc_empty0 + 8 * buf, ((chunk / kTcAccBufs) & 1) ^ 1);
            TCP(st_acc += clock64() - tq;)
            d_tmem = tmem_base + (uint32_t)(buf * kTcNMax);
            acc = 0;
          }
          TCP(tq = clock64();)
          mbar_wait(b_full(sb), pb);
          if (PAIR) mbar_wait(b_fwd(sb), pb);          // ... and the peer's half
          TCP(st_b += clock64() - tq;)
          tc_fence_after();
          TCP(tq = clock64();)
          // descriptors advance by plain 64-bit adds on the (address >> 4) field: no re-encoding per MMA
          uint64_t da = a_desc0 + (uint64_t)e.tap;                                  // tap j = window shifted by j rows of 16 B
          uint64_t db = tc_desc(b_base + (uint32_t)sb * b_stage_bytes, b_lbo, 128);
          const uint64_t b_lo_off = (uint64_t)((PAIR ? 1u : 2u) * e.nks * N);      // (kbs / 4) * N (pair: N/2) * 16 bytes >> 4
          const int nks = no_mma ? 0 : e.nks;
          // all TF32 MMAs of the stage, then all BF16 correction MMAs (same accumulator, order is free): alternating the
          // MMA kind instruction by instruction cost ~12 clk per MMA
#pragma unroll 4
          for (int ks = 0; ks < nks; ++ks) {
            if (leader) {
              if (PAIR) tc_mma2_tf32(d_tmem, da, db, idesc, acc);
              else tc_mma_tf32(d_tmem, da, db, idesc, acc);                                       // a_hi * b_hi
            }
            acc = 1;
            da += a_ks; db += b_ks;
          }
          if (terms >= 2) {
            da = a_desc0 + (uint64_t)e.tap + a_lo_off;
            db = tc_desc(b_base + (uint32_t)sb * b_stage_bytes, b_lbo, 128) + b_lo_off;
#pragma unroll 4
            for (int ks = 0; ks < nks; ++ks) {
              if (leader) {
                if (PAIR) tc_mma2_bf16(d_tmem, da, db, idesc16);
                else tc_mma_bf16(d_tmem, da, db, idesc16);                                        // a_lo * b_hi + a_hi * b_lo
              }
              da += a_ks; db += b_ks;
            }
          }
          if (leader) {
            if (PAIR) {
              tc_commit2(b_empty(sb));
              if (e.flags & kTcChunkLast) tc_commit2(acc_full0 + 8 * (chunk % kTcAccBufs));
              if (e.flags & kTcKbLast) tc_commit2(a_empty(sa));
            } else {
              tc_commit(b_empty(sb));
              if (e.flags & kTcChunkLast) tc_commit(acc_full0 + 8 * (chunk % kTcAccBufs));
              if (e.flags & kTcKbLast) tc_commit(a_empty(sa));
            }
          }
          __syncwarp();
          TCP(st_issue += clock64() - tq;)
          if (++sb == NBS) { sb = 0; pb ^= 1; }
          if (e.flags & kTcChunkLast) ++chunk;
          if (e.flags & kTcKbLast) { if (++sa == kTcAStages) { sa = 0; pa ^= 1; } }
        }
      }
#ifdef AVC_TC_PROFILE
      if ((p.dbg & 32) && blockIdx.x == 0 && lane == 0)
        printf("[conv_tc cta0] issuer: total %lld clk, wait a_full %lld, wait b_full %lld, wait acc_empty %lld, issue %lld (items %d)\n",
               clock64() - t_begin, st_a, st_b, st_acc, st_issue, (n_work + (int)gridDim.x - 1) / (int)gridDim.x);
#endif
#undef TCP
    }
  } else if (warp < 6) {
    // ===== loaders (128 threads): window gather + TF32 split =====
    // Thread tl owns window row tl (8 float4 per K block); the <= 7 rows past 128 are spread one float4
    // per thread.  The loads of K block kb+1 are issued right after K block kb is stored, so they fly
    // while the thread waits for the stage to be released.
    pdl_wait();
    const int tl = threadIdx.x - 64;   // 0..127
    const int er = tl >> 3, ec = tl & 7;   // my share of the extra rows: row 128 + er, chunk ec
    int sa = 0; uint32_t pa = 0;
    const bool skip = (p.dbg & 2) != 0;
#ifdef AVC_TC_PROFILE
    long long l_setup = 0, l_wait = 0, l_store = 0, l_fetch = 0, l_t0 = clock64(), lq;
#define TCL(x) x
#else
#define TCL(x)
#endif
    for (int wk = w_first; wk < n_work; wk += w_step) {
      const TcPass& ps = p.pass[wk % p.n_pass];
      const long long v0 = tile_row0(wk);
      for (int gi = ps.g_begin; gi < ps.g_end; ++gi) {
        TCL(lq = clock64();)
        const TcGroup& G = p.g[gi];
        const float* src[2]; const float* msk[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int i = j == 0 ? tl : kTcM + er;
          src[j] = nullptr; msk[j] = nullptr;
          if (j == 0 || er < G.n_taps - 1) {
            const long long u = v0 + i;
            const int b = (int)(u / p.Pv);
            const int pos = G.sg * (int)(u - (long long)b * p.Pv) + G.off0;
            int rr = pos;
            if constexpr (VL) {
              rr = tc_src_row_vl(p, b, pos);
              if (rr >= 0 && !skip) {
                src[j] = p.A + (long long)b * p.a_bs + (long long)rr * p.a_rs + G.a_ch_off;
                if (p.Mk) msk[j] = p.Mk + (long long)b * p.m_bs + (long long)rr * p.m_rs + G.a_ch_off;
              }
            } else {
              if (!p.bwd) {
                rr = rr < 0 ? -rr : rr;
                if (rr >= p.T_a) rr = 2 * (p.T_a - 1) - rr;
              }
              if (b < p.B && rr >= 0 && rr < p.T_a && !skip) {
                src[j] = p.A + (long long)b * p.a_bs + (long long)rr * p.a_rs + G.a_ch_off;
                if (p.Mk) msk[j] = p.Mk + (long long)b * p.m_bs + (long long)rr * p.m_rs + G.a_ch_off;
              }
            }
          }
        }
        const bool have_e = er < G.n_taps - 1;
        const int nkb = (G.kc + kTcKB - 1) / kTcKB;
        float4 v[kTcKB / 4], m[kTcKB / 4], ve, me;
        auto fetch = [&](int kb) {
          const int kb0 = kb * kTcKB, kbs = min(kTcKB, G.kc - kb0);
#pragma unroll
          for (int c = 0; c < kTcKB / 4; ++c) v[c] = (src[0] && 4 * c < kbs) ? ld4(src[0] + kb0 + 4 * c) : f4zero();
          ve = (src[1] && 4 * ec < kbs) ? ld4(src[1] + kb0 + 4 * ec) : f4zero();
          if (p.Mk) {
#pragma unroll
            for (int c = 0; c < kTcKB / 4; ++c) m[c] = (msk[0] && 4 * c < kbs) ? ld4(msk[0] + kb0 + 4 * c) : f4zero();
            me = (msk[1] && 4 * ec < kbs) ? ld4(msk[1] + kb0 + 4 * ec) : f4zero();
          }
        };
        // L2 prefetch runs kTcPfDist K blocks ahead of the register fetch (one 128-byte line per row and K block)
        auto prefetch = [&](int kb) {
          if (kb >= nkb) return;
          const int kb0 = kb * kTcKB;
          if (src[0]) { prefetch_l2(src[0] + kb0); if (msk[0]) prefetch_l2(msk[0] + kb0); }
          if (ec == 0 && src[1]) { prefetch_l2(src[1] + kb0); if (msk[1]) prefetch_l2(msk[1] + kb0); }
        };
#pragma unroll 1
        for (int d = 1; d <= kTcPfDist; ++d) prefetch(d);
        TCL(l_setup += clock64() - lq;)
        // kb = -1 only fetches K block 0; afterwards: store K block kb, then issue the loads of kb + 1 so that they
        // fly while this thread waits for the next stage to be released (one fetch site: code size matters here)
#pragma unroll 1
        for (int kb = -1; kb < nkb; ++kb) {
          if (kb >= 0) {
            const int kbs = min(kTcKB, G.kc - kb * kTcKB);
            TCL(lq = clock64();)
            mbar_wait(a_empty(sa), pa ^ 1);
            TCL(l_wait += clock64() - lq; lq = clock64();)
            float* hi = As + (size_t)sa * 2 * kTcAPlane;
            float* lo = hi + kTcAPlane;
            if (p.Mk) {
#pragma unroll
              for (int c = 0; c < kTcKB / 4; ++c) v[c] = dact4mul(v[c], m[c], p.slope);
              ve = dact4mul(ve, me, p.slope);
            }
            // plane 0: TF32 hi parts [k/4][row][4 floats]; plane 1: per k-step of 8 channels two 16-byte K chunks per row,
            // bf16(lo[0..8)) then bf16(hi[0..8)) -- the K = 16 operand of the correction MMA (pairs with the weights' hi|lo chunks)
#pragma unroll
            for (int ks = 0; ks < kTcKB / 8; ++ks) {
              if (8 * ks >= kbs) break;
              const float4 a = v[2 * ks], b = v[2 * ks + 1];
              const float4 ha = make_float4(tf32_hi(a.x), tf32_hi(a.y), tf32_hi(a.z), tf32_hi(a.w));
              const float4 hb = make_float4(tf32_hi(b.x), tf32_hi(b.y), tf32_hi(b.z), tf32_hi(b.w));
              st4(hi + ((size_t)(2 * ks) * kTcRows + tl) * 4, ha);
              st4(hi + ((size_t)(2 * ks + 1) * kTcRows + tl) * 4, hb);
              st_bf16x8(lo + ((size_t)(2 * ks) * kTcRows + tl) * 4, f4sub(a, ha), f4sub(b, hb));
              st_bf16x8(lo + ((size_t)(2 * ks + 1) * kTcRows + tl) * 4, ha, hb);
            }
            if (have_e && 4 * ec < kbs) {   // extra rows: this thread holds 4 of the 8 channels of its k-step
              const float4 h = make_float4(tf32_hi(ve.x), tf32_hi(ve.y), tf32_hi(ve.z), tf32_hi(ve.w));
              st4(hi + ((size_t)ec * kTcRows + kTcM + er) * 4, h);
              float* q = lo + ((size_t)(ec & ~1) * kTcRows + kTcM + er) * 4 + 2 * (ec & 1);
              st_bf16x4(q, f4sub(ve, h));
              st_bf16x4(q + (size_t)kTcRows * 4, h);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { if (PAIR) mbar_arrive_cta(a_full(sa), 0); else mbar_arrive(a_full(sa)); }
            TCL(l_store += clock64() - lq; lq = clock64();)
            if (++sa == kTcAStages) { sa = 0; pa ^= 1; }
          }
          if (kb + 1 < nkb) fetch(kb + 1);
          prefetch(kb + 1 + kTcPfDist);
          TCL(if (kb >= 0) l_fetch += clock64() - lq;)
        }
      }
    }
#ifdef AVC_TC_PROFILE
    if ((p.dbg & 32) && blockIdx.x == 0 && tl == 0)
      printf("[conv_tc cta0] loader: total %lld clk, setup %lld, wait a_empty %lld, split+store %lld, fetch issue %lld\n",
             clock64() - l_t0, l_setup, l_wait, l_store, l_fetch);
#endif
#undef TCL
  } else {
    // ===== drain warps (256 threads): chunk sums in registers, then the epilogue =====
    pdl_wait();
    int chunk = 0;
    TcDrainProf dp{0, 0, 0};
    TCD(const long long d_t0 = clock64();)
    for (int wk = w_first; wk < n_work; wk += w_step) {
      const TcPass& ps = p.pass[wk % p.n_pass];
      const long long v0 = tile_row0(wk);
      float* scratch = scr_all + (size_t)(warp - 6) * 32 * kTcScrPitch;
      tc_drain_and_store<VL>(p, ps, tmem_base, acc_full0, acc_empty0, v0, warp, lane, chunk, scratch, dp, PAIR ? 0 : -1);
    }
#ifdef AVC_TC_PROFILE
    if ((p.dbg & 32) && blockIdx.x == 0 && warp == 6 && lane == 0)
      printf("[conv_tc cta0] drain: total %lld clk, wait acc_full %lld, tmem ld+add %lld, epilogue %lld (chunks %d)\n",
             clock64() - d_t0, dp.wait, dp.ld, dp.epi, chunk);
#endif
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();      // the leader's MMAs write the peer's TMEM and read its shared memory: leave together
  if (warp == 0) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// dgrad: add the extended rows (gradient of the reflect padding) to their mirror rows.
//   row r' in [1, PL]        += side[PL - r']
//   row r' in [T-1-PR, T-2]  += side[PL + T - 2 - r']          (both scaled by act'(Om) like the main rows)
// VL: T is utterance b's own length, lens[b]
template <bool VL = false>
__global__ void tc_fold_kernel(float* __restrict__ Y, long long y_bs, int y_rs, const float* __restrict__ side,
                               const float* __restrict__ Om, long long om_bs, int om_rs, float slope,
                               int B, int T_max, int N, int PL, int PR, const int* __restrict__ lens) {
  pdl_enter();
  const int n4 = N >> 2, H = PL + PR;
  const long long tot = (long long)B * H * n4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % n4) << 2;
    const long long bj = i / n4;
    const int j = (int)(bj % H), b = (int)(bj / H);
    const int T = VL ? lens[b] : T_max;
    const int r = j < PL ? j + 1 : T - 1 - PR + (j - PL);
    if (r < 0 || r >= T) continue;
    if (j >= PL && r >= 1 && r <= PL) continue;                 // the left-edge thread of this row adds both parts
    const float* sb = side + (long long)b * H * N + c;
    float4 a = f4zero();
    if (r >= 1 && r <= PL) a = f4add(a, ld4(sb + (long long)(PL - r) * N));
    if (r >= T - 1 - PR && r <= T - 2) a = f4add(a, ld4(sb + (long long)(PL + T - 2 - r) * N));
    if (Om) a = dact4mul(a, ld4(Om + (long long)b * om_bs + (long long)r * om_rs + c), slope);
    float* y = Y + (long long)b * y_bs + (long long)r * y_rs + c;
    st4(y, f4add(ld4(y), a));
  }
}

inline size_t tc_smem_bytes() {
  return (size_t)kTcAStages * 2 * kTcAPlane * 4 + (size_t)kTcBStages * 2 * (kTcKB / 4) * kTcNMax * 16 + kTcBarSlots * 8 + (size_t)8 * 32 * kTcScrPitch * 4;
}

// ---- host: the tensor-core view of one conv launch (passes x groups, no tensor pointers yet) --------
struct TcOp {
  int n_pass = 0, n_groups = 0;
  int kmax = 1;          // most taps of any group
  int sdiv = 1;          // dgrad: virtual rows advance sdiv output rows (conv stride)
  int n_out = 0;         // total output columns
  TcPass pass[kTcMaxPass];
  TcGroup g[kTcMaxPass];
  bool add_pass(int g_begin, int g_end, int N, int ch_off, int so, int oo) {
    if (n_pass >= kTcMaxPass) return false;
    pass[n_pass++] = TcPass{g_begin, g_end, N, ch_off, so, oo};
    return true;
  }
  int add_group(const float* Wp, int a_ch_off, int kc, int n_taps, int sg, int off0) {
    if (n_groups >= kTcMaxPass) return -1;
    g[n_groups] = TcGroup{Wp, a_ch_off, kc, n_taps, sg, off0};
    kmax = std::max(kmax, n_taps);
    return n_groups++;
  }
};

inline int tc_stage_count(const TcOp& op) {
  int n = 0;
  for (int q = 0; q < op.n_pass; ++q)
    for (int g = op.pass[q].g_begin; g < op.pass[q].g_end; ++g) n += ((op.g[g].kc + kTcKB - 1) / kTcKB) * op.g[g].n_taps;
  return n;
}

inline bool tc_supported(const ConvArgs& a, const TcOp& op) {
  if (op.n_pass <= 0 || op.n_groups <= 0) return false;
  if (tc_stage_count(op) > kTcMaxStages) return false;
  if (a.Y2 && a.bwd) return false;
  if (a.res.mode != RES_NONE && (a.res.rf < 1 || a.res.rf > 2)) return false;   // the epilogue reads at most two skip rows per output row
  if (a.Om && a.res.mode != RES_NONE) return false;                              // one set of operand registers serves either
  for (int g = 0; g < op.n_groups; ++g)
    if (!op.g[g].Wp || op.g[g].kc % 8 || op.g[g].a_ch_off % 4 || op.g[g].n_taps < 1 || op.g[g].n_taps > kMaxTaps) return false;
  for (int q = 0; q < op.n_pass; ++q)
    if (op.pass[q].N != 128 && op.pass[q].N != 80) return false;
  if (a.a_rs % 4 || (a.Mk && a.m_rs % 4)) return false;
  return true;
}

inline void tc_halo(const ConvArgs& a, int& PL, int& PR) {
  PL = PR = 0;
  if (a.bwd) for (int g = 0; g < a.n_groups; ++g) { PL = std::max(PL, a.g[g].pl); PR = std::max(PR, a.g[g].pr); }
}

// side: scratch of tc_side_floats(a) floats for dgrad (nullptr for forward)
inline size_t tc_side_floats(const ConvArgs& a) {
  int PL, PR;
  tc_halo(a, PL, PR);
  return (size_t)a.B * (PL + PR) * a.N;
}

inline TcArgs tc_make_args(const ConvArgs& a, const TcOp& op, float* side, int terms) {
  TcArgs t{};
  t.A = a.A; t.a_bs = a.a_bs; t.a_rs = a.a_rs; t.T_a = a.T_a;
  t.Mk = a.Mk; t.m_bs = a.m_bs; t.m_rs = a.m_rs; t.slope = a.slope;
  t.bwd = a.bwd;
  int PL, PR;
  tc_halo(a, PL, PR);
  t.T_y = a.T_y; t.halo_l = PL; t.halo_r = PR;
  const int n_valid = a.bwd ? (a.T_y + PL + PR + op.sdiv - 1) / op.sdiv : a.T_y;
  t.Pv = n_valid + op.kmax - 1;
  t.B = a.B; t.Mv = (long long)a.B * t.Pv;
  t.side_n = a.N;
  t.Y = a.Y; t.y_bs = a.y_bs; t.y_rs = a.y_rs;
  t.Y2 = a.Y2; t.y2_bs = a.y2_bs; t.y2_rs = a.y2_rs;
  t.bias = a.bias; t.act = a.act;
  t.Om = a.Om; t.om_bs = a.om_bs; t.om_rs = a.om_rs;
  t.res = a.res;
  t.side = (PL + PR) > 0 ? side : nullptr;
  t.n_pass = op.n_pass;
  t.terms = terms;
  { static const int cs = getenv("AVC_TC_CHUNK") ? atoi(getenv("AVC_TC_CHUNK")) : kTcChunkSteps; t.chunk_steps = cs; }
  { static const int dbg = getenv("AVC_TC_DBG") ? atoi(getenv("AVC_TC_DBG")) : 0; t.dbg = dbg; }
  for (int g = 0; g < op.n_groups; ++g) t.g[g] = op.g[g];
  // stage table: (group, K block, tap) in the order every role visits them; an accumulation chunk closes after the
  // tap that brings it to chunk_steps MMA k-steps and after the last tap of the pass
  int ns = 0;
  for (int q = 0; q < op.n_pass; ++q) {
    TcPass ps = op.pass[q];
    ps.s_begin = ns; ps.n_chunks = 0;
    int steps = 0;
    for (int g = ps.g_begin; g < ps.g_end; ++g) {
      const TcGroup& G = op.g[g];
      const int nkb = (G.kc + kTcKB - 1) / kTcKB;
      for (int kb = 0; kb < nkb; ++kb) {
        const int kbs = std::min(kTcKB, G.kc - kb * kTcKB);
        for (int tap = 0; tap < G.n_taps; ++tap) {
          if (ns >= kTcMaxStages) fail(AVC_ERR_STATE, "conv_tc: stage table overflow (tc_supported should have refused this conv)");
          TcStage& e = t.st[ns++];
          e.w_off = (uint32_t)((size_t)kb * G.n_taps * 2 * kTcKB * ps.N + (size_t)tap * 2 * kbs * ps.N);
          e.gi = (uint8_t)g; e.tap = (uint8_t)tap; e.nks = (uint8_t)(kbs / 8);
          unsigned fl = 0;
          if (tap == 0) fl |= kTcKbFirst;
          if (tap == G.n_taps - 1) fl |= kTcKbLast;
          if (steps == 0) fl |= kTcChunkFirst;
          steps += kbs / 8;
          const bool last = g == ps.g_end - 1 && kb == nkb - 1 && tap == G.n_taps - 1;
          if (last || steps >= t.chunk_steps) { fl |= kTcChunkLast; steps = 0; ++ps.n_chunks; }
          e.flags = (uint8_t)fl;
        }
      }
    }
    ps.s_end = ns;
    t.pass[q] = ps;
  }
  return t;
}

}  // namespace avc
