// conv_tc2.cuh -- the tcgen05 implicit-GEMM Conv1d with the operand roles SWAPPED: weights are the M = 128 operand, 256 window
// rows are the N operand, the accumulator in TMEM is the TRANSPOSED output tile D^T[c_out][row].
//
// Why (scripts/ubench/mma_shapes.cu, profiles/r02a_mma_shapes.txt, measured on B200):
//   * one thread issues tcgen05.mma and the tensor pipe keeps only about two instructions in flight: every cycle the issuing
//     thread spends between two MMAs on barrier waits, fences and descriptor arithmetic beyond the length of ONE MMA is a cycle
//     the pipe idles.  With N = 128 an MMA is 64 clk and the per-stage protocol of conv_tc.cuh (two mbarrier waits, a commit)
//     costs 119 clk per MMA in isolation (112-131 in the kernel) against a floor of 64.7; switching kind::tf32 <-> kind::f16
//     costs another ~64 clk at N = 128 and nothing at N = 256.
//   * operand fetch is NOT the limit: N = 128 and N = 256 both run at the 64.7 clk per 128x128x8 floor back to back, with 100
//     B/clk of concurrent STS, 160 B/clk of LDS and bulk copies in the background; 128-byte swizzle and A-from-TMEM change nothing.
//   So: N = 256 MMAs (128 clk each: twice the cover for the same protocol) -- c_out is 128 in this model, hence the swap --
//   and fewer waits per MMA (the weight ring is handed over per 4-MMA plane, the window per K block).
//
// What else the transposed tile buys: a drain lane owns one output CHANNEL and 128 consecutive rows, so the epilogue stores
// straight from registers with lanes along the channel axis (128 B per warp and row, coalesced) -- no shared-memory transpose.
//
// Same numerics as conv_tc.cuh (same split, same packed weight images, same chunked accumulation, same stage table).
//   warp 0      weight producer: one bulk copy (TMA engine, mbarrier complete_tx) per 16 KB plane of a stage, ring of 5
//   warp 1      MMA issuer
//   warps 2-7   window loaders (192 threads): (row, k-step) units of 32 B, row pointers in a shared-memory table
//   warps 8-15  drain (TMEM -> fp32 chunk sums in registers) + epilogue; setmaxnreg gives them 160 registers, the rest 96
#pragma once
#include <type_traits>

#include "conv_tc.cuh"

namespace avc {

constexpr int kT2N = 256;                         // window rows (GEMM N) of one tile
constexpr int kT2Rows = kT2N + kMaxTaps;          // rows of one window stage
constexpr int kT2XStages = 2;
constexpr int kT2WSlots = 5;                      // weight ring, in planes (half stages) of 16 KB
constexpr int kT2Threads = 512;
constexpr int kT2Loaders = 192;
constexpr int kT2XPlane = (kTcKB / 4) * kT2Rows * 4;              // floats of one plane of a window stage
constexpr int kT2WPlaneBytes = (kTcKB / 4) * kTcNMax * 16;        // 16 KB
constexpr int kT2AccBufs = 2;                                     // 2 x 256 TMEM columns

inline size_t tc2_smem_bytes() {
  return (size_t)kT2XStages * 2 * kT2XPlane * 4 + (size_t)kT2WSlots * kT2WPlaneBytes + 32 * 8 + (size_t)2 * kT2Rows * 8 + (size_t)kT2N * 5 * 4;
}

// ---- epilogue ------------------------------------------------------------------------------------
// Row descriptors: everything that depends on the virtual row (utterance, output row, skip rows and their weight) is worked out
// ONCE per tile, one row per drain thread, and kept in shared memory as element offsets (five arrays of kT2N words); the epilogue
// reads them with broadcast LDS.  (Every lane of every drain warp needs every row's addresses: computing them per lane would
// cost a 64-bit division per row and lane.)  The epilogue itself is branch-free straight-line code -- predicated stores, the
// operand loads of eight rows in flight before the first is consumed: the first version branched per row (dead / halo / main)
// and ran one row at a time behind an LDS -> branch -> STG chain, 25-60k clk per tile (profiles/r02b_conv_tc2_roles.txt).
constexpr int kT2DescWords = 5;     // yoff | y2off | g0 | g1 | rs
// yoff: -1 dead row, <= -2: dgrad halo row at side-buffer offset -2 - yoff; g0 / g1: -1 = none

template <bool VL>
__device__ __forceinline__ void t2_make_desc(const TcArgs& p, const TcPass& ps, long long u, int* __restrict__ tab, int row) {
  const TcRow r = tc_row<VL>(p, ps, u);
  int yoff = -1, y2off = 0, g0 = -1, g1 = -1;
  if (r.kind == 2) yoff = -2 - (int)(((long long)r.b * (p.halo_l + p.halo_r) + r.o) * p.side_n);
  if (r.kind == 1) {
    yoff = (int)((long long)r.b * p.y_bs + (long long)r.o * p.y_rs);
    if (p.Y2) y2off = (int)((long long)r.b * p.y2_bs + (long long)r.o * p.y2_rs);
    if (p.Om) g0 = (int)((long long)r.b * p.om_bs + (long long)r.o * p.om_rs);
    else if (p.res.mode != RES_NONE) {
      g0 = (int)((long long)r.b * p.res.bs + (long long)r.t0 * p.res.rs);
      if (r.t1 >= 0) g1 = (int)((long long)r.b * p.res.bs + (long long)r.t1 * p.res.rs);
    }
  }
  tab[row] = yoff; tab[kT2N + row] = y2off; tab[2 * kT2N + row] = g0; tab[3 * kT2N + row] = g1; tab[4 * kT2N + row] = __float_as_int(r.rs);
}

// plain (non-volatile) shared loads: the descriptors are read-only while an epilogue runs, so the compiler may batch and hoist
// them; `base` is produced by a volatile asm AFTER the barrier that publishes the table, which keeps them below it
__device__ __forceinline__ int t2_lds(uint32_t addr) { int v; asm("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }

// predicated store without a branch around the arithmetic that feeds it: rows stay independent instruction streams
__device__ __forceinline__ void t2_st_if(float* ptr, float v, bool ok) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.global.f32 [%0], %1;\n\t}" ::"l"(ptr), "f"(v), "r"((int)ok));
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// MODE: 0 plain, 1 act' mask on the output (Om), 2 one skip row (RES_SAME / RES_UP / RES_POOL_BWD), 3 two skip rows (RES_POOL / RES_UP_BWD)
// HALO: dgrad launches whose extended rows go to the side buffer.
// The finished sums are read back from TMEM eight rows at a time in a ROLLED loop (t_sum: this warp's 32 lanes x 128 columns):
// a fully unrolled epilogue over 128 accumulator registers is 28 KB of straight-line code per variant that every drain warp
// executes exactly once per tile, and it ran at the speed of instruction fetch (10-58k clk per tile, profiles/r02b_conv_tc2_roles.txt).
template <int MODE, bool HALO>
__device__ __forceinline__ void t2_epilogue(const TcArgs& p, uint32_t t_sum, uint32_t tab, int c, bool c_ok) {
  const float bias = (p.bias && c_ok) ? p.bias[c] : 0.f;
  const float* G = MODE == 1 ? p.Om : p.res.R;
  float* const Y = p.Y + c;
  float* const Y2 = p.Y2 ? p.Y2 + c : nullptr;
  float* const S = HALO ? p.side + c : nullptr;
  const bool act = p.act != 0, has_y2 = p.Y2 != nullptr;
  const float slope = p.slope;
  // rows whose operand loads are in flight before the first is consumed: the sums wait in TMEM, so the registers are free
  // for 32 (two-operand modes: 16) rows of operands -- 8 drain warps x 32 loads cover the ~1k clk of an L2 / HBM round trip
  constexpr int NB = MODE == 3 ? 16 : 32;
#pragma unroll 1
  for (int r0 = 0; r0 < 128; r0 += NB) {
    uint32_t v[NB];
#pragma unroll
    for (int j = 0; j < NB; j += 16) tmem_ld16(t_sum + r0 + j, *reinterpret_cast<uint32_t(*)[16]>(&v[j]));
    float ga[NB], gb[NB];
    if (MODE >= 1) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        const int g0 = t2_lds(tab + 4 * (2 * kT2N + r0 + j));
        ga[j] = 0.f; gb[j] = 0.f;
        if (c_ok && g0 >= 0) ga[j] = G[g0 + c];
        if (MODE == 3) {
          const int g1 = t2_lds(tab + 4 * (3 * kT2N + r0 + j));
          if (c_ok && g1 >= 0) gb[j] = G[g1 + c];
        }
      }
    }
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int yo = t2_lds(tab + 4 * (r0 + j));
      const float raw = __uint_as_float(v[j]);
      float x = raw + bias;
      if (MODE == 1) x *= (ga[j] > 0.f ? 1.f : slope);
      x = (act && !(x > 0.f)) ? x * slope : x;
      const bool main_row = c_ok && yo >= 0;
      if (MODE >= 2) {
        if (has_y2) t2_st_if(Y2 + t2_lds(tab + 4 * (kT2N + r0 + j)), x, main_row);
        const float rs = __int_as_float(t2_lds(tab + 4 * (4 * kT2N + r0 + j)));
        x += (MODE == 3 ? ga[j] + gb[j] : ga[j]) * rs;
      }
      if (HALO) {
        const bool halo_row = c_ok && yo < -1;
        t2_st_if(halo_row ? S + (-2 - yo) : Y + yo, halo_row ? raw : x, main_row || halo_row);
      } else {
        t2_st_if(Y + yo, x, main_row);
      }
    }
  }
}

// VL = true: ragged batch, lengths from p.lens_* (see TcArgs).
template <bool VL = false>
__global__ void __launch_bounds__(kT2Threads, 1) conv_tc2_kernel(const TcArgs p) {
  extern __shared__ __align__(128) unsigned char t2_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Xs = reinterpret_cast<float*>(t2_smem);                                              // [2 stages][2 planes][kT2XPlane]
  unsigned char* Ws = t2_smem + (size_t)kT2XStages * 2 * kT2XPlane * 4;                        // [5 slots][16 KB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ws + (size_t)kT2WSlots * kT2WPlaneBytes);
  long long* rowtab = reinterpret_cast<long long*>(bars + 32);                                 // [2][kT2Rows]: element offsets of the window rows (A, mask)
  int* desc = reinterpret_cast<int*>(rowtab + 2 * kT2Rows);                                   // [kT2DescWords][kT2N] output row descriptors of the current tile
  const uint32_t bar0 = smem_u32(bars);
  auto x_full = [&](int s) { return bar0 + 8 * s; };
  auto x_empty = [&](int s) { return bar0 + 8 * (2 + s); };
  auto w_full = [&](int s) { return bar0 + 8 * (4 + s); };
  auto w_empty = [&](int s) { return bar0 + 8 * (9 + s); };
  const uint32_t acc_full0 = bar0 + 8 * 14, acc_empty0 = bar0 + 8 * 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kT2XStages; ++s) { mbar_init(x_full(s), kT2Loaders / 32); mbar_init(x_empty(s), 1); }
    for (int s = 0; s < kT2WSlots; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), 1); }
    for (int s = 0; s < kT2AccBufs; ++s) { mbar_init(acc_full0 + 8 * s, 1); mbar_init(acc_empty0 + 8 * s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();

  const int n_tiles = (int)((p.Mv + kT2N - 1) / kT2N);
  const int n_work = n_tiles * p.n_pass;
  const int w_first = (int)blockIdx.x, w_step = (int)gridDim.x;

  if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
    if (warp == 0) {
      // ===== weight producer =====
      if (lane == 0) {
        int sw = 0; uint32_t pw = 0;
        for (int wk = w_first; wk < n_work; wk += w_step) {
          const TcPass& ps = p.pass[wk % p.n_pass];
          const uint32_t N = (uint32_t)ps.N;
#pragma unroll 1
          for (int s = ps.s_begin; s < ps.s_end; ++s) {
            const TcStage e = p.st[s];
            const uint32_t bytes = 32u * e.nks * N;                  // ONE plane: 8 nks channels x N x 4 bytes
            const float* src = p.g[e.gi].Wp + e.w_off;
#pragma unroll 1
            for (int u = 0; u < 2; ++u) {
              mbar_wait(w_empty(sw), pw ^ 1);
              mbar_expect_tx(w_full(sw), bytes);
              bulk_g2s(smem_u32(Ws + (size_t)sw * kT2WPlaneBytes), src + (size_t)u * (bytes >> 2), bytes, w_full(sw));
              if (++sw == kT2WSlots) { sw = 0; pw ^= 1; }
            }
          }
        }
      }
    } else if (warp == 1) {
      // ===== MMA issuer: the whole warp walks the table, one elected lane issues =====
      const bool leader = elect_one();
      int sx = 0, sw = 0; uint32_t px = 0, pw = 0;
      int chunk = 0;
      const int terms = p.terms;
#ifdef AVC_TC_PROFILE
      long long st_x = 0, st_w = 0, st_acc = 0, st_issue = 0, t_begin = clock64(), tq;   // build with -DAVC_TC_PROFILE, run with AVC_TC_DBG=32
#define T2P(x) x
#else
#define T2P(x)
#endif
      const uint32_t x_base = smem_u32(Xs), w_base = smem_u32(Ws);
      constexpr uint32_t x_lbo = kT2Rows * 16;
      constexpr uint64_t x_ks = (uint64_t)((2 * x_lbo) >> 4), x_lo_off = (uint64_t)((kT2XPlane * 4) >> 4);
      for (int wk = w_first; wk < n_work; wk += w_step) {
        const TcPass& ps = p.pass[wk % p.n_pass];
        const uint32_t N = (uint32_t)ps.N;                                                       // valid output channels (M is always 128)
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kT2N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t idesc16 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kT2N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t w_lbo = N * 16;
        const uint64_t w_ks = (uint64_t)((2 * w_lbo) >> 4);
        uint64_t x_desc0 = 0;
        uint32_t d_tmem = 0, acc = 0;
#pragma unroll 1
        for (int s = ps.s_begin; s < ps.s_end; ++s) {
          const TcStage e = p.st[s];
          if (e.flags & kTcKbFirst) {
            T2P(tq = clock64();)
            mbar_wait(x_full(sx), px);
            T2P(if (st_issue == 0) t_begin = clock64(); else st_x += clock64() - tq;)
            x_desc0 = tc_desc(x_base + (uint32_t)sx * (2 * kT2XPlane * 4), x_lbo, 128);
          }
          if (e.flags & kTcChunkFirst) {
            const int buf = chunk % kT2AccBufs;
            T2P(tq = clock64();)
            mbar_wait(acc_empty0 + 8 * buf, ((chunk / kT2AccBufs) & 1) ^ 1);
            T2P(st_acc += clock64() - tq;)
            d_tmem = tmem_base + (uint32_t)(buf * kT2N);
            acc = 0;
          }
          const int nks = e.nks;
          // plane 0: kind::tf32  D^T += W_hi * X_hi^T
          T2P(tq = clock64();)
          mbar_wait(w_full(sw), pw);
          T2P(st_w += clock64() - tq; tq = clock64();)
          tc_fence_after();
          {
            uint64_t dw = tc_desc(w_base + (uint32_t)sw * kT2WPlaneBytes, w_lbo, 128);
            uint64_t dx = x_desc0 + (uint64_t)e.tap;
#pragma unroll 4
            for (int ks = 0; ks < nks; ++ks) {
              if (leader) tc_mma_tf32(d_tmem, dw, dx, idesc, acc);
              acc = 1;
              dw += w_ks; dx += x_ks;
            }
            if (leader) tc_commit(w_empty(sw));
            if (++sw == kT2WSlots) { sw = 0; pw ^= 1; }
          }
          // plane 1: kind::f16 (bf16, K = 16)  D^T += [W_hi | W_lo] * [X_lo | X_hi]^T
          T2P(st_issue += clock64() - tq; tq = clock64();)
          mbar_wait(w_full(sw), pw);
          T2P(st_w += clock64() - tq; tq = clock64();)
          tc_fence_after();
          {
            uint64_t dw = tc_desc(w_base + (uint32_t)sw * kT2WPlaneBytes, w_lbo, 128);
            uint64_t dx = x_desc0 + (uint64_t)e.tap + x_lo_off;
            if (terms >= 2) {
#pragma unroll 4
              for (int ks = 0; ks < nks; ++ks) {
                if (leader) tc_mma_bf16(d_tmem, dw, dx, idesc16);
                dw += w_ks; dx += x_ks;
              }
            }
            if (leader) {
              tc_commit(w_empty(sw));
              if (e.flags & kTcChunkLast) tc_commit(acc_full0 + 8 * (chunk % kT2AccBufs));
              if (e.flags & kTcKbLast) tc_commit(x_empty(sx));
            }
            if (++sw == kT2WSlots) { sw = 0; pw ^= 1; }
          }
          __syncwarp();
          T2P(st_issue += clock64() - tq;)
          if (e.flags & kTcChunkLast) ++chunk;
          if (e.flags & kTcKbLast) { if (++sx == kT2XStages) { sx = 0; px ^= 1; } }
        }
      }
#ifdef AVC_TC_PROFILE
      if ((p.dbg & 32) && blockIdx.x == 0 && lane == 0)
        printf("[conv_tc2 cta0] issuer: total %lld clk, wait x_full %lld, wait w_full %lld, wait acc_empty %lld, issue %lld (items %d)\n",
               clock64() - t_begin, st_x, st_w, st_acc, st_issue, (n_work + (int)gridDim.x - 1) / (int)gridDim.x);
#endif
    } else {
      // ===== window loaders (192 threads) =====
      // unit q of a K block = (row q / 4, k-step q % 4): four consecutive lanes read the 128 contiguous bytes of one row's
      // 32 channels; every thread handles units tl, tl + 192, ... (5.5 on average), three at a time.
      pdl_wait();
      const int tl = threadIdx.x - 64;                    // 0..191
      int sx = 0; uint32_t px = 0;
#ifdef AVC_TC_PROFILE
      long long l_wait = 0, l_tab = 0, l_t0 = clock64(), lq;
#endif
      for (int wk = w_first; wk < n_work; wk += w_step) {
        const TcPass& ps = p.pass[wk % p.n_pass];
        const long long v0 = (long long)(wk / p.n_pass) * kT2N;
        for (int gi = ps.g_begin; gi < ps.g_end; ++gi) {
          const TcGroup& G = p.g[gi];
          const int n_rows = kT2N + G.n_taps - 1;
          // row table: element offset of every window row in A (and in the mask tensor), -1 = zeros
          T2P(lq = clock64();)
          asm volatile("bar.sync 1, %0;" ::"r"(kT2Loaders) : "memory");          // the previous group's readers are done
          for (int i = tl; i < n_rows; i += kT2Loaders) {
            const long long u = v0 + i;
            const int b = (int)(u / p.Pv);
            const int pos = G.sg * (int)(u - (long long)b * p.Pv) + G.off0;
            int rr = pos;
            bool ok;
            if constexpr (VL) {
              rr = tc_src_row_vl(p, b, pos);
              ok = rr >= 0;
            } else {
              if (!p.bwd) {
                rr = rr < 0 ? -rr : rr;
                if (rr >= p.T_a) rr = 2 * (p.T_a - 1) - rr;
              }
              ok = b < p.B && rr >= 0 && rr < p.T_a;
            }
            rowtab[i] = ok ? (long long)b * p.a_bs + (long long)rr * p.a_rs + G.a_ch_off : -1;
            rowtab[kT2Rows + i] = (ok && p.Mk) ? (long long)b * p.m_bs + (long long)rr * p.m_rs + G.a_ch_off : -1;
          }
          asm volatile("bar.sync 1, %0;" ::"r"(kT2Loaders) : "memory");
          T2P(l_tab += clock64() - lq;)
          const int nkb = (G.kc + kTcKB - 1) / kTcKB;
          const int n_units = n_rows * 4;
          const bool masked = p.Mk != nullptr;
          // L2 prefetch kTcPfDist K blocks ahead: one 128-byte line per row and K block (lanes with ks == 0)
          auto prefetch = [&](int kb) {
            if (kb >= nkb) return;
            for (int q = tl; q < n_units; q += kT2Loaders)
              if ((q & 3) == 0) {
                const long long o = rowtab[q >> 2];
                if (o >= 0) { prefetch_l2(p.A + o + kb * kTcKB); if (masked) prefetch_l2(p.Mk + rowtab[kT2Rows + (q >> 2)] + kb * kTcKB); }
              }
          };
#pragma unroll 1
          for (int d = 0; d < kTcPfDist; ++d) prefetch(d);
#pragma unroll 1
          for (int kb = 0; kb < nkb; ++kb) {
            const int kb0 = kb * kTcKB, kbs = min(kTcKB, G.kc - kb0);
            prefetch(kb + kTcPfDist);
            float* hi = Xs + (size_t)sx * 2 * kT2XPlane;
            float* lo = hi + kT2XPlane;
            bool waited = false;
            // NU units per round: every load of a round is in flight before the first is consumed (and, for the first round,
            // before the thread waits for the stage to be released)
            auto round = [&](auto nu_tag, int q0) {
              constexpr int NU = decltype(nu_tag)::value;
              float4 va[NU], vb[NU], ma[NU > 3 ? 1 : NU], mb[NU > 3 ? 1 : NU];
#pragma unroll
              for (int j = 0; j < NU; ++j) {
                const int q = q0 + j * kT2Loaders;
                va[j] = f4zero(); vb[j] = f4zero();
                if (NU <= 3) { ma[j] = f4zero(); mb[j] = f4zero(); }
                if (q < n_units) {
                  const int ks = q & 3;
                  const long long o = rowtab[q >> 2];
                  if (o >= 0 && 8 * ks < kbs) {
                    const float* src = p.A + o + kb0 + 8 * ks;
                    va[j] = ld4(src); vb[j] = ld4(src + 4);
                    if (NU <= 3) { const float* ms = p.Mk + rowtab[kT2Rows + (q >> 2)] + kb0 + 8 * ks; ma[j] = ld4(ms); mb[j] = ld4(ms + 4); }
                  }
                }
              }
              if (!waited) { T2P(lq = clock64();) mbar_wait(x_empty(sx), px ^ 1); waited = true; T2P(l_wait += clock64() - lq;) }
#pragma unroll
              for (int j = 0; j < NU; ++j) {
                const int q = q0 + j * kT2Loaders;
                if (q < n_units) {
                  const int ks = q & 3, row = q >> 2;
                  if (8 * ks < kbs) {
                    float4 a = va[j], b = vb[j];
                    if (NU <= 3) { a = dact4mul(a, ma[j], p.slope); b = dact4mul(b, mb[j], p.slope); }
                    const float4 ha = make_float4(tf32_hi(a.x), tf32_hi(a.y), tf32_hi(a.z), tf32_hi(a.w));
                    const float4 hb = make_float4(tf32_hi(b.x), tf32_hi(b.y), tf32_hi(b.z), tf32_hi(b.w));
                    st4(hi + ((size_t)(2 * ks) * kT2Rows + row) * 4, ha);
                    st4(hi + ((size_t)(2 * ks + 1) * kT2Rows + row) * 4, hb);
                    st_bf16x8(lo + ((size_t)(2 * ks) * kT2Rows + row) * 4, f4sub(a, ha), f4sub(b, hb));
                    st_bf16x8(lo + ((size_t)(2 * ks + 1) * kT2Rows + row) * 4, ha, hb);
                  }
                }
              }
            };
            if (masked) {
#pragma unroll 1
              for (int q0 = tl; q0 < n_units; q0 += 3 * kT2Loaders) round(std::integral_constant<int, 3>{}, q0);
            } else {
#pragma unroll 1
              for (int q0 = tl; q0 < n_units; q0 += 6 * kT2Loaders) round(std::integral_constant<int, 6>{}, q0);
            }
            if (!waited) mbar_wait(x_empty(sx), px ^ 1);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(x_full(sx));
            if (++sx == kT2XStages) { sx = 0; px ^= 1; }
          }
        }
      }
#ifdef AVC_TC_PROFILE
      if ((p.dbg & 32) && blockIdx.x == 0 && tl == 0)
        printf("[conv_tc2 cta0] loader: total %lld clk, row tables %lld, wait x_empty %lld\n", clock64() - l_t0, l_tab, l_wait);
#endif
    }
  } else {
    // ===== drain warps (256 threads): chunk sums in registers, then the epilogue straight from registers =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
    pdl_wait();
    const int quad = warp & 3, half = (warp - 8) >> 2;
    const int dt = threadIdx.x - 256;                   // 0..255: the tile row whose descriptor this thread works out
    int chunk = 0;
#ifdef AVC_TC_PROFILE
    long long d_wait = 0, d_ld = 0, d_epi = 0, d_desc = 0, d_t0 = clock64(), dq;
#endif
    int mode = 0;
    if (p.Om) mode = 1;
    else if (p.res.mode == RES_POOL || p.res.mode == RES_UP_BWD) mode = 3;
    else if (p.res.mode != RES_NONE) mode = 2;
    if (p.side) mode += 4;
    for (int wk = w_first; wk < n_work; wk += w_step) {
      const TcPass& ps = p.pass[wk % p.n_pass];
      const long long v0 = (long long)(wk / p.n_pass) * kT2N;
      const int cl = quad * 32 + lane;                  // channel within the pass (TMEM lane)
      const bool c_ok = cl < ps.N;
      const bool q_ok = quad * 32 < ps.N;               // this warp's lanes hold any valid channel at all
      // ---- row descriptors of this tile (while the first chunk's MMAs run) ----
      T2P(dq = clock64();)
      asm volatile("bar.sync 2, 256;" ::: "memory");    // the previous tile's epilogue has read its descriptors
      {
        t2_make_desc<VL>(p, ps, v0 + dt, desc, dt);
        const int g0 = desc[2 * kT2N + dt], g1 = desc[3 * kT2N + dt];
        if (kTcPfDist > 0 && g0 >= 0) {                 // the epilogue's operands for this row: into L2 now, read ~20k clk later
          const float* G = p.Om ? p.Om : p.res.R;
          for (int c0 = 0; c0 < ps.N; c0 += 32) {
            prefetch_l2(G + g0 + ps.ch_off + c0);
            if (g1 >= 0) prefetch_l2(G + g1 + ps.ch_off + c0);
          }
        }
      }
      asm volatile("bar.sync 2, 256;" ::: "memory");
      uint32_t tab;
      asm volatile("mov.u32 %0, %1;" : "=r"(tab) : "r"(smem_u32(desc) + (uint32_t)(half * 128 * 4)) : "memory");   // descriptor loads stay below the barrier
      T2P(d_desc += clock64() - dq;)
      float acc[128];
#pragma unroll
      for (int i = 0; i < 128; ++i) acc[i] = 0.f;
      uint32_t t_sum = 0;
      int last_buf = 0;
#pragma unroll 1
      for (int cc = 0; cc < ps.n_chunks; ++cc) {
        const int buf = chunk % kT2AccBufs;
        const bool last = cc == ps.n_chunks - 1;
        T2P(dq = clock64();)
        mbar_wait(acc_full0 + 8 * buf, (chunk / kT2AccBufs) & 1);
        T2P(d_wait += clock64() - dq; dq = clock64();)
        tc_fence_after();
        const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * kT2N + half * 128);
        if (q_ok) {
#pragma unroll
          for (int c0 = 0; c0 < 128; c0 += 32) {
            uint32_t r0[16], r1[16];
            tmem_ld16(t0 + c0, r0);
            tmem_ld16(t0 + c0 + 16, r1);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) { acc[c0 + i] += __uint_as_float(r0[i]); acc[c0 + 16 + i] += __uint_as_float(r1[i]); }
            if (last) { tmem_st16(t0 + c0, &acc[c0]); tmem_st16(t0 + c0 + 16, &acc[c0 + 16]); }     // the finished sums go back in place
          }
        }
        ++chunk;
        if (last) { t_sum = t0; last_buf = buf; break; }       // this buffer is released after the epilogue has read it
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty0 + 8 * buf);
        T2P(d_ld += clock64() - dq;)
      }
      T2P(dq = clock64();)
      if (q_ok) {
        tmem_st_wait();
        const int c = ps.ch_off + cl;
        switch (mode) {      // one specialised epilogue per launch
          case 0: t2_epilogue<0, false>(p, t_sum, tab, c, c_ok); break;
          case 1: t2_epilogue<1, false>(p, t_sum, tab, c, c_ok); break;
          case 2: t2_epilogue<2, false>(p, t_sum, tab, c, c_ok); break;
          case 3: t2_epilogue<3, false>(p, t_sum, tab, c, c_ok); break;
          case 4: t2_epilogue<0, true>(p, t_sum, tab, c, c_ok); break;
          case 5: t2_epilogue<1, true>(p, t_sum, tab, c, c_ok); break;
          case 6: t2_epilogue<2, true>(p, t_sum, tab, c, c_ok); break;
          default: t2_epilogue<3, true>(p, t_sum, tab, c, c_ok); break;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty0 + 8 * last_buf);
      T2P(d_epi += clock64() - dq;)
    }
#ifdef AVC_TC_PROFILE
    if ((p.dbg & 32) && blockIdx.x == 0 && warp == 8 && lane == 0)
      printf("[conv_tc2 cta0] drain: total %lld clk, descriptors %lld, wait acc_full %lld, tmem ld+add %lld, epilogue %lld (chunks %d, mode %d)\n",
             clock64() - d_t0, d_desc, d_wait, d_ld, d_epi, chunk, mode);
#endif
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

}  // namespace avc
