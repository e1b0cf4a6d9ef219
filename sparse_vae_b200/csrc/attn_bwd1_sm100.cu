// Block-sparse attention backward for sm_100a in ONE pass over the sequence (tcgen05 / TMEM / TMA): every tensor is
// read once and written once (8 units of HBM traffic, the algorithmic minimum of SURVEY 8d), nothing is accumulated
// with atomics, and S / P never reach HBM.
//
// Work decomposition.  The B*H*ceil(L/128) key tiles are cut into one contiguous range per CTA (one persistent CTA per
// SM); inside a range a "segment" is a run of consecutive key tiles kt = t0 .. t1-1 of one (batch, head) sequence.
// The CTA walks a segment in order.  For key tile kt (key blocks 4kt+c, c = 0..3 = TMEM lane quarter) the causal band
// of width `left` makes query blocks 4kt .. 4kt+left+2 attend it ("slots" i = 0 .. nq-1, nq = left+3 <= 7), so
//   dK, dV of the tile are COMPLETE after the tile (accumulated in TMEM over its slots), while
//   dQ of query tile kt receives the slots 0-3 of key tile kt and the slots 4-6 of key tile kt-1.
// dQ therefore lives in two TMEM accumulators that swap roles from tile to tile: X (query tile kt: finished and
// stored at the end of tile kt) and Y (query tile kt+1: started by tile kt).  A segment that does not start at the
// beginning of its sequence first runs a "pre-tile" (key tile t0-1, slots 4-6 only, nothing stored) that rebuilds the
// Y contribution it would otherwise have to fetch from another CTA -- no cross-CTA exchange, bit-deterministic.
// The GLOBAL key block 0 (include_cls) is attended by every query: key tile kt handles it against its own 128
// queries in query-major form (S_g = Q K_0^T), adds dS_g K_0 to dQ X and accumulates [dO^T ; Q^T] [P_g | dS_g]
// (= dV_0^T and dK_0^T) over the whole segment in a fifth accumulator, written as an fp32 partial at the end of the
// segment; `attn_bwd_finish_kernel` sums a sequence's partials in a fixed order.
//
// Per tile the work is a stream of "units" (one 32-query slot, or the global block): S^T = K Q_i^T and dP^T = V dO_i^T
// (128 keys x 32 queries each) into the 64-column TMEM score buffer of one of two math warpgroups -> the group pulls
// the scores into registers (the buffer is free for the next S^T at once), computes
// P^T = exp2(S^T*scale*log2e - lse*log2e), dS^T = P^T o (dP^T - delta) * scale, writes both as 16-bit into its 32-column
// TMEM operand buffer (A operands of dV += P^T dO_i and dK += dS^T Q_i) and dS^T also into shared memory, from where
// dQ (+)= dS K (A MN-major from shared memory, 4 slots = 128 queries at a time) is issued.  16 warps:
//   warps 0-3 / 4-7   math warpgroups (even / odd units; warp = TMEM lane quarter = key block)
//   warps 8-11        epilogue group: accumulators -> 16-bit -> shared memory -> TMA store; delta = rowsum(dO o O)
//                     and -lse*log2e of every arriving query tile (O read straight from global memory)
//   warp 12           TMA producer (K / V double-buffered, Q / dO in a 3-deep ring of query tiles)
//   warp 13           tcgen05.mma issuer: S^T / dP^T, as soon as the owning group has emptied its score buffer
//   warp 14           tcgen05.mma issuer: dV, dK (A from TMEM)
//   warp 15           tcgen05.mma issuer: dQ X / Y, the global block's dQ and dK_0 / dV_0 products
// TMEM (512 columns): dK 0 | dV 64 | dQ 128 / 192 | G 256 | score buffers 320 / 384 | 16-bit operand buffers 448 / 480.
//
// Reference: autograd of sdd -> softmax -> dsd, sparse_vae/core/sparse_matmul.py:463-488 (dV = P^T dO, dP = dO V^T,
// dQ = dS K, dK = dS^T Q) and the block-sparse softmax backward dS = P o (dP - rowsum(dP o P)) * scale.
// Roofline: HBM-bound; algorithmic bytes = 8 * B*L*H*Dh * 2 (read Q,K,V,O,dO; write dQ,dK,dV).
#include <type_traits>

#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kB1Threads = 512;
constexpr int kB1MaxLeft = 4;

template <int DH>
struct B1Smem {
  static constexpr int ROWB = DH * 2;
  static constexpr int TILE = kTile * ROWB;                 // 16 KB
  static constexpr int SLOT = kBlock * ROWB;                // 4 KB
  static constexpr int OFF_RING = 0;                        // [3] x { dO tile | Q tile }: the stacked operand [dO^T ; Q^T]
  static constexpr int OFF_K = OFF_RING + 3 * 2 * TILE;     // [2] K tile (later the dK staging tile)
  static constexpr int OFF_V = OFF_K + 2 * TILE;            // [2]
  static constexpr int OFF_DS = OFF_V + 2 * TILE;           // dS^T of 4 slots: 2 halves x [128 keys][64 queries]
  static constexpr int OFF_G = OFF_DS + 2 * TILE;           // [128 queries][P_g (32 keys) | dS_g (32 keys)]
  static constexpr int OFF_K0 = OFF_G + TILE;               // key block 0
  static constexpr int OFF_V0 = OFF_K0 + SLOT;
  static constexpr int OFF_STAT = OFF_V0 + SLOT;            // [3][2][128] fp32: -lse*log2e, -delta*scale per ring tile
  static constexpr int OFF_KPM0 = OFF_STAT + 3 * 2 * kTile * 4;   // [32] fp32: additive mask of key block 0 (log2 domain)
  static constexpr int OFF_BAR = OFF_KPM0 + 256;            // (+ 32 zeros after the mask values)
  static constexpr int NBAR = 40;
  static constexpr int DYN_BYTES = OFF_BAR + NBAR * 8 + 16 + 1024;
  static constexpr int COL_DK = 0, COL_DV = 64, COL_DQ = 128, COL_G = 256, COL_U = 320, COL_A = 448;
  static_assert(DYN_BYTES <= 227 * 1024, "shared memory");
};

struct B1Params {
  const float* kpm;        // [B, L] additive or null
  const float* lse;        // [B, H, L]
  const void* out;         // O, read directly (delta)
  int64_t o_stride[3];     // {batch, head, row} in elements
  float* gpart;            // [B*H][maxseg][2 (dK, dV)][32 keys][DH] fp32 partials of the global key block
  int maxseg;
  int L, H, T, nb;         // T = key / query tiles per sequence
  int left, cls, nq;       // band width, global column, slots per key tile (left + 3)
  int num_tiles, num_ctas;
  float scale, scale_log2;
};

// first tile of CTA i's range
__host__ __device__ inline int b1_range_lo(int i, int num_tiles, int num_ctas) {
  return (int)(((long long)i * num_tiles) / num_ctas);
}
// the CTA whose range holds tile x
__host__ __device__ inline int b1_cta_of(int x, int num_tiles, int num_ctas) {
  int i = (int)(((long long)x * num_ctas) / num_tiles);
  if (i >= num_ctas) i = num_ctas - 1;
  while (i + 1 < num_ctas && b1_range_lo(i + 1, num_tiles, num_ctas) <= x) ++i;
  while (i > 0 && b1_range_lo(i, num_tiles, num_ctas) > x) --i;
  return i;
}

// ---- the unit stream of a segment, enumerated identically by every role -------------------------------------
struct B1Seg {
  int seq, b, h, t0, t1;
  int kfirst;        // first key tile processed (t0 - 1 when a pre-tile is needed)
  int ntiles;        // processed tiles including the pre-tile
  int has_pre;
  int nqt;           // query tiles loaded: t0 .. t0 + nqt - 1
  int gslot;         // index of this segment's partial of the global key block
};

struct B1Geom {
  int nq, cls, nx, XU, NU, halo, T;
  __device__ B1Geom(const B1Params& p) {
    nq = p.nq; cls = p.cls; T = p.T;
    nx = nq < 4 ? nq : 4;            // slots of group X (query tile kt)
    XU = nx + cls;                   // units of group X including the global block
    NU = nq + cls;
    halo = nq > 4;                   // slots 4.. exist: query tile kt+1 is touched
  }
  // local tile j of the segment -> key tile, unit positions [ub, ue)
  __device__ void tile(const B1Seg& s, int j, int& kt, bool& pre, int& ub, int& ue) const {
    kt = s.kfirst + j;
    pre = s.has_pre && j == 0;
    ub = pre ? XU : 0;
    ue = (halo && kt + 1 < T) ? NU : XU;
  }
  // does a tile whose units end at `ue` contribute slots 4.. to the next query tile (group Y)?
  __device__ bool has_y(int ue) const { return halo && ue == NU; }
  // unit position -> slot (-1: the global block)
  __device__ int slot_of(int pos) const {
    if (pos < nx) return pos;
    if (cls && pos == nx) return -1;
    return pos - cls;
  }
};

__device__ inline B1Seg b1_make_seg(const B1Params& p, const B1Geom& g, int start, int end) {
  B1Seg s;
  s.seq = start / p.T;
  s.b = s.seq / p.H;
  s.h = s.seq % p.H;
  s.t0 = start % p.T;
  const int room = p.T - s.t0;
  s.t1 = s.t0 + ((end - start) < room ? (end - start) : room);
  s.has_pre = (g.halo && s.t0 > 0) ? 1 : 0;
  s.kfirst = s.t0 - s.has_pre;
  s.ntiles = s.t1 - s.kfirst;
  const int last_q = (g.halo && s.t1 < p.T) ? s.t1 : s.t1 - 1;
  s.nqt = last_q - s.t0 + 1;
  s.gslot = (int)blockIdx.x - b1_cta_of(s.seq * p.T, p.num_tiles, p.num_ctas);
  return s;
}

// barrier indices
enum : int {
  BAR_K_FULL = 0,      // [2] TMA -> S^T issuer
  BAR_V_FULL = 2,      // [2]
  BAR_Q_FULL = 4,      // [3] TMA -> S^T issuer, epilogue group (statistics)
  BAR_STAT = 7,        // [3] epilogue group -> math groups: statistics of the ring tile (one arrival per warp)
  BAR_S_READY = 10,    // [2] S^T issuer -> math group                                           (per group)
  BAR_P_READY = 13,    // [2] math group -> dV/dK issuer (band units) or dQ issuer (global unit)   (one arrival per warp)
  BAR_U_FREE = 16,     // [2] the group has the scores in registers -> S^T issuer                 (one arrival per warp)
  BAR_A_FREE = 34,     // [2] the MMAs that read the group's 16-bit operands have retired -> math group
  BAR_GRPX_READY = 19, // dS^T of every slot of group X (0-3) is in shared memory -> dQ issuer      (4 warps x 4 slots)
  BAR_DS_FREE = 20,    // dQ MMAs have read the dS^T staging tile -> math groups
  BAR_G_FREE = 21,     // the global block's products have read sG -> math groups
  BAR_ACC_READY = 22,  // all dV / dK MMAs of the tile retired -> epilogue group
  BAR_ACC_FREE = 23,   // epilogue has read the accumulators -> dV/dK issuer                               (one arrival per warp)
  BAR_K_FREE = 24,     // [2] epilogue -> TMA
  BAR_V_FREE = 26,     // [2] S^T issuer -> TMA
  BAR_RING_FREE = 28,  // [3] epilogue -> TMA
  BAR_K0_FULL = 31,
  BAR_GRPY_READY = 32, // same for group Y (slots 4..)                                                (4 warps x (nq - 4) slots)
  BAR_ACC_READY2 = 33, // all dQ / global-block MMAs of the tile retired -> epilogue group
  BAR_COUNT = 36
};

__device__ __forceinline__ void mbar_inval(uint64_t* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <typename T, int DH>
__global__ void __launch_bounds__(kB1Threads, 1)
attn_bwd1_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                       const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                       const __grid_constant__ CUtensorMap tmK32, const __grid_constant__ CUtensorMap tmV32,
                       const __grid_constant__ CUtensorMap tmDQ, const __grid_constant__ CUtensorMap tmDK,
                       const __grid_constant__ CUtensorMap tmDV, const B1Params p) {
  static_assert(DH == 64, "the stacked [dO^T ; Q^T] operand and the 128-byte rows need head_dim 64");
  using S = B1Smem<DH>;
  constexpr int ROWB = S::ROWB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + S::NBAR);
  float* sStat = reinterpret_cast<float*>(smem + S::OFF_STAT);
  float* sKpm0 = reinterpret_cast<float*>(smem + S::OFF_KPM0);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const B1Geom g(p);

  auto init_barriers = [&]() {
    auto init_n = [&](int first, int n, uint32_t count) { for (int i = 0; i < n; ++i) mbar_init(bars + first + i, count); };
    init_n(BAR_K_FULL, 2, 1); init_n(BAR_V_FULL, 2, 1); init_n(BAR_Q_FULL, 3, 1); init_n(BAR_STAT, 3, 4);
    init_n(BAR_S_READY, 2, 1); init_n(BAR_P_READY, 2, 4); init_n(BAR_U_FREE, 2, 4); init_n(BAR_A_FREE, 2, 1); init_n(BAR_GRPX_READY, 1, 4 * g.nx);
    init_n(BAR_GRPY_READY, 1, 4 * (g.halo ? g.nq - 4 : 1));
    init_n(BAR_DS_FREE, 1, 1); init_n(BAR_G_FREE, 1, 1); init_n(BAR_ACC_READY, 1, 1); init_n(BAR_ACC_READY2, 1, 1);
    init_n(BAR_ACC_FREE, 1, 4);
    init_n(BAR_K_FREE, 2, 1); init_n(BAR_V_FREE, 2, 1); init_n(BAR_RING_FREE, 3, 1); init_n(BAR_K0_FULL, 1, 1);
    fence_barrier_init();
  };

  if (threadIdx.x == 0) init_barriers();
  if (warp == 15) {
    if (lane == 0) {
      prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV);
      prefetch_tensormap(&tmK32); prefetch_tensormap(&tmV32); prefetch_tensormap(&tmDQ); prefetch_tensormap(&tmDK);
      prefetch_tensormap(&tmDV);
    }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int range_lo = b1_range_lo(blockIdx.x, p.num_tiles, p.num_ctas);
  const int range_hi = b1_range_lo(blockIdx.x + 1, p.num_tiles, p.num_ctas);

  // Between two segments: everything of the finished segment has retired (CTA-wide barrier), then the mbarriers are
  // re-created, so that every segment starts with all phases at zero and local counters.
  auto segment_sync = [&]() {
    tc_fence_before();
    named_bar_sync(15, kB1Threads);
    if (threadIdx.x == 0) {
      for (int i = 0; i < BAR_COUNT; ++i) mbar_inval(bars + i);
      init_barriers();
    }
    named_bar_sync(15, kB1Threads);
    tc_fence_after();
  };

  auto ring_do = [&](int n) { return smem + S::OFF_RING + (n % 3) * 2 * S::TILE; };               // dO tile of local query tile n
  auto ring_q = [&](int n) { return smem + S::OFF_RING + (n % 3) * 2 * S::TILE + S::TILE; };      // Q tile

  if (warp >= 12) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 12) {
      // ============================================== TMA producer ==============================================
      for (int start = range_lo; start < range_hi;) {
        const B1Seg s = b1_make_seg(p, g, start, range_hi);
        start += s.t1 - s.t0;
        if (g.cls) {
          mbar_arrive_expect_tx_w(bars + BAR_K0_FULL, 2 * S::SLOT);
          tma_load_4d_w(smem + S::OFF_K0, &tmK32, bars + BAR_K0_FULL, 0, 0, s.h, s.b);
          tma_load_4d_w(smem + S::OFF_V0, &tmV32, bars + BAR_K0_FULL, 0, 0, s.h, s.b);
        }
        int qnext = 0;
        for (int j = 0; j < s.ntiles; ++j) {
          int kt, ub, ue;
          bool pre;
          g.tile(s, j, kt, pre, ub, ue);
          const int sl = j & 1;
          if (j >= 2) mbar_wait(bars + BAR_V_FREE + sl, ((j - 2) >> 1) & 1);
          mbar_arrive_expect_tx_w(bars + BAR_V_FULL + sl, S::TILE);
          tma_load_4d_w(smem + S::OFF_V + sl * S::TILE, &tmV, bars + BAR_V_FULL + sl, 0, kt * kTile, s.h, s.b);
          if (j >= 2) mbar_wait(bars + BAR_K_FREE + sl, ((j - 2) >> 1) & 1);
          mbar_arrive_expect_tx_w(bars + BAR_K_FULL + sl, S::TILE);
          tma_load_4d_w(smem + S::OFF_K + sl * S::TILE, &tmK, bars + BAR_K_FULL + sl, 0, kt * kTile, s.h, s.b);
          // query tiles this key tile touches: kt (local kt - t0; not for the pre-tile) and kt + 1 (slots 4..)
          int need = g.has_y(ue) ? (kt + 1 - s.t0) + 1 : (kt - s.t0) + 1;
          if (need > s.nqt) need = s.nqt;
          for (; qnext < need; ++qnext) {
            const int n = qnext, r = n % 3;
            if (n >= 3) mbar_wait(bars + BAR_RING_FREE + r, ((n - 3) / 3) & 1);
            mbar_arrive_expect_tx_w(bars + BAR_Q_FULL + r, 2 * S::TILE);
            tma_load_4d_w(ring_do(n), &tmDO, bars + BAR_Q_FULL + r, 0, (s.t0 + n) * kTile, s.h, s.b);
            tma_load_4d_w(ring_q(n), &tmQ, bars + BAR_Q_FULL + r, 0, (s.t0 + n) * kTile, s.h, s.b);
          }
        }
        segment_sync();
      }
    } else if (warp == 13) {
      // ============================================== S^T / dP^T issuer =========================================
      const uint32_t idesc_s = make_idesc(kTile, kBlock, Elem<T>::fmt, 0, 0);
      const uint32_t k0_addr = smem_u32(smem + S::OFF_K0), v0_addr = smem_u32(smem + S::OFF_V0);
      for (int start = range_lo; start < range_hi;) {
        const B1Seg s = b1_make_seg(p, g, start, range_hi);
        start += s.t1 - s.t0;
        int u = 0, q_waited = 0;
        bool k0_waited = false;
        for (int j = 0; j < s.ntiles; ++j) {
          int kt, ub, ue;
          bool pre;
          g.tile(s, j, kt, pre, ub, ue);
          const int sl = j & 1;
          const uint32_t k_addr = smem_u32(smem + S::OFF_K + sl * S::TILE), v_addr = smem_u32(smem + S::OFF_V + sl * S::TILE);
          mbar_wait(bars + BAR_K_FULL + sl, (j >> 1) & 1);
          mbar_wait(bars + BAR_V_FULL + sl, (j >> 1) & 1);
          for (int pos = ub; pos < ue; ++pos, ++u) {
            const int buf = u & 1;                                           // = the math group that owns the unit
            const int slot = g.slot_of(pos);
            const int n = (kt - s.t0) + (slot < 0 ? 0 : (slot >> 2));       // local query tile of the unit
            for (; q_waited <= n; ++q_waited) mbar_wait(bars + BAR_Q_FULL + q_waited % 3, (q_waited / 3) & 1);
            if (slot < 0 && !k0_waited) { mbar_wait(bars + BAR_K0_FULL, 0); k0_waited = true; }
            if (u >= 2) mbar_wait(bars + BAR_U_FREE + buf, ((u - 2) >> 1) & 1);
            tc_fence_after();
            const uint32_t d_s = tmem_base + S::COL_U + 64 * buf, d_dp = d_s + 32;
            const uint32_t q_addr = smem_u32(ring_q(n)), do_addr = smem_u32(ring_do(n));
            uint32_t a_s, b_s, a_dp, b_dp;
            if (slot >= 0) {       // S^T = K Q_i^T, dP^T = V dO_i^T
              a_s = k_addr; b_s = q_addr + (slot & 3) * S::SLOT; a_dp = v_addr; b_dp = do_addr + (slot & 3) * S::SLOT;
            } else {               // S_g = Q K_0^T, dP_g = dO V_0^T (query-major)
              a_s = q_addr; b_s = k0_addr; a_dp = do_addr; b_dp = v0_addr;
            }
#pragma unroll
            for (int ks = 0; ks < DH / 16; ++ks) {
              mma_ss_w(d_s, make_smem_desc(a_s + ks * 32, 16, 8 * ROWB, ROWB), make_smem_desc(b_s + ks * 32, 16, 8 * ROWB, ROWB),
                       idesc_s, ks > 0 ? 1u : 0u);
              mma_ss_w(d_dp, make_smem_desc(a_dp + ks * 32, 16, 8 * ROWB, ROWB), make_smem_desc(b_dp + ks * 32, 16, 8 * ROWB, ROWB),
                       idesc_s, ks > 0 ? 1u : 0u);
            }
            tc_commit_w(bars + BAR_S_READY + buf);
          }
          tc_commit_w(bars + BAR_V_FREE + sl);         // every MMA that reads this V tile has been issued
        }
        segment_sync();
      }
    } else if (warp == 14) {
      // ============================================== dV / dK issuer ============================================
      const uint32_t idesc_o = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
      for (int start = range_lo; start < range_hi;) {
        const B1Seg s = b1_make_seg(p, g, start, range_hi);
        start += s.t1 - s.t0;
        int u = 0;
        for (int j = 0; j < s.ntiles; ++j) {
          int kt, ub, ue;
          bool pre;
          g.tile(s, j, kt, pre, ub, ue);
          uint32_t acc = 0;
          for (int pos = ub; pos < ue; ++pos, ++u) {
            const int buf = u & 1;
            const int slot = g.slot_of(pos);
            mbar_wait(bars + BAR_P_READY + buf, (u >> 1) & 1);      // every phase is observed, in order
            if (slot < 0) continue;                     // the global unit's MMAs belong to warp 15
            if (!pre) {
              // (the epilogue arrives once per tile, pre-tiles included: it has then seen the previous tile's
              //  ACC_READY / ACC_READY2 phases, so those barriers can never run two phases ahead of their waiter)
              if (acc == 0 && j >= 1) mbar_wait(bars + BAR_ACC_FREE, (j - 1) & 1);
              tc_fence_after();
              const int n = (kt - s.t0) + (slot >> 2);
              const uint32_t q_addr = smem_u32(ring_q(n)) + (slot & 3) * S::SLOT, do_addr = smem_u32(ring_do(n)) + (slot & 3) * S::SLOT;
              const uint32_t ta = tmem_base + S::COL_A + 32 * buf;
#pragma unroll
              for (int k2 = 0; k2 < 2; ++k2) {          // dV += P^T dO_i ; dK += dS^T Q_i   (16 queries per MMA)
                mma_ts_w(tmem_base + S::COL_DV, ta + 8 * k2, make_smem_desc(do_addr + k2 * 16 * ROWB, S::SLOT, 8 * ROWB, ROWB),
                         idesc_o, acc);
                mma_ts_w(tmem_base + S::COL_DK, ta + 16 + 8 * k2, make_smem_desc(q_addr + k2 * 16 * ROWB, S::SLOT, 8 * ROWB, ROWB),
                         idesc_o, acc);
                acc = 1;
              }
            }
            tc_commit_w(bars + BAR_A_FREE + buf);
          }
          tc_commit_w(bars + BAR_ACC_READY);
        }
        segment_sync();
      }
    } else {
      // ============================================== dQ / global-block issuer ==================================
      const uint32_t idesc_o = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);      // A from TMEM, B MN-major
      const uint32_t idesc_mn = make_idesc(kTile, DH, Elem<T>::fmt, 1, 1);     // A and B MN-major, N = 64
      const uint32_t ds_addr = smem_u32(smem + S::OFF_DS), g_addr = smem_u32(smem + S::OFF_G);
      const uint32_t k0_addr = smem_u32(smem + S::OFF_K0);
      for (int start = range_lo; start < range_hi;) {
        const B1Seg s = b1_make_seg(p, g, start, range_hi);
        start += s.t1 - s.t0;
        int u = 0, xgroups = 0, ygroups = 0, gtiles = 0;
        bool prev_y = false;                 // the previous tile left its slots 4.. in this tile's X accumulator
        for (int j = 0; j < s.ntiles; ++j) {
          int kt, ub, ue;
          bool pre;
          g.tile(s, j, kt, pre, ub, ue);
          const uint32_t k_addr = smem_u32(smem + S::OFF_K + (j & 1) * S::TILE);
          const uint32_t acc_x = tmem_base + S::COL_DQ + 64 * (kt & 1), acc_y = tmem_base + S::COL_DQ + 64 * ((kt + 1) & 1);
          // dQ (+)= dS K over the 128 keys of the tile: A = staged dS^T read MN-major (two 64-query halves 16 KB apart)
          auto issue_dq = [&](uint32_t d, uint32_t first_acc, uint64_t* ready, int& count) {
            mbar_wait(ready, count & 1);
            ++count;
            tc_fence_after();
#pragma unroll
            for (int k2 = 0; k2 < kTile / 16; ++k2)
              mma_ss_w(d, make_smem_desc(ds_addr + k2 * 16 * 128, S::TILE, 8 * 128, 128),
                       make_smem_desc(k_addr + k2 * 16 * ROWB, S::SLOT, 8 * ROWB, ROWB), idesc_mn, k2 > 0 ? 1u : first_acc);
            tc_commit_w(bars + BAR_DS_FREE);
          };
          for (int pos = ub; pos < ue; ++pos, ++u) {
            const int buf = u & 1;
            const int slot = g.slot_of(pos);
            if (slot == g.nx - 1) issue_dq(acc_x, prev_y ? 1u : 0u, bars + BAR_GRPX_READY, xgroups);
            if (slot >= 4 && slot == g.nq - 1) issue_dq(acc_y, 0u, bars + BAR_GRPY_READY, ygroups);
            if (slot < 0) {
              mbar_wait(bars + BAR_P_READY + buf, (u >> 1) & 1);
              tc_fence_after();
              const int n = kt - s.t0;
              const uint32_t do_addr = smem_u32(ring_do(n));
              const uint32_t ta = tmem_base + S::COL_A + 32 * buf;
#pragma unroll
              for (int k2 = 0; k2 < 2; ++k2)            // dQ X += dS_g K_0
                mma_ts_w(acc_x, ta + 8 * k2, make_smem_desc(k0_addr + k2 * 16 * ROWB, S::SLOT, 8 * ROWB, ROWB), idesc_o, 1u);
              // G (+)= [dO^T ; Q^T] (128 x 128 queries) [P_g | dS_g] (128 queries x 64): rows 0-63 x columns 0-31 = dV_0^T,
              // rows 64-127 x columns 32-63 = dK_0^T
#pragma unroll
              for (int k2 = 0; k2 < kTile / 16; ++k2)
                mma_ss_w(tmem_base + S::COL_G, make_smem_desc(do_addr + k2 * 16 * ROWB, S::TILE, 8 * ROWB, ROWB),
                         make_smem_desc(g_addr + k2 * 16 * 128, 16 * 128, 8 * 128, 128), idesc_mn, (k2 > 0 || gtiles > 0) ? 1u : 0u);
              tc_commit_w(bars + BAR_A_FREE + buf);
              tc_commit_w(bars + BAR_G_FREE);
              ++gtiles;
            }
          }
          tc_commit_w(bars + BAR_ACC_READY2);
          prev_y = g.has_y(ue);
        }
        segment_sync();
      }
    }
  } else if (warp >= 8) {
    // ================================================ epilogue group ===============================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
    const int w = warp & 3;
    const int tid_g = threadIdx.x & 127;
    const int row = w * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(w * 32) << 16);

    const T* __restrict__ O = reinterpret_cast<const T*>(p.out);

    for (int start = range_lo; start < range_hi;) {
      const B1Seg s = b1_make_seg(p, g, start, range_hi);
      start += s.t1 - s.t0;
      const int64_t stat_base = ((int64_t)s.b * p.H + s.h) * p.L;
      const T* o_seq = O + (int64_t)s.b * p.o_stride[0] + (int64_t)s.h * p.o_stride[1];

      // -lse*log2e and -delta*scale of local query tile n, delta = rowsum(dO o O): 8 lanes per row (16 bytes each),
      // O straight from global memory (coalesced 128-byte rows), dO from the ring tile.  Two halves: the global loads
      // are issued early (stats_issue) and consumed after the accumulators of the current tile have been drained --
      // the drain comes first because the next tile's dV / dK MMAs wait for it.  (Measured alternatives: statistics
      // before the drain 207 us instead of 190 us; statistics in the otherwise idle TMA producer warp 506 us -- one
      // warp cannot hide the latency of the global loads.)
      const int chunk = tid_g & 7, rsub = tid_g >> 3;
      uint4 ov[8];
      float lv[8];
      auto stats_issue = [&](int n) {
        const int q0 = (s.t0 + n) * kTile;
#pragma unroll
        for (int ps = 0; ps < 8; ++ps) {
          const int qpos = q0 + ps * 16 + rsub;
          ov[ps] = make_uint4(0, 0, 0, 0);
          lv[ps] = 0.f;
          if (qpos < p.L) {
            ov[ps] = __ldg(reinterpret_cast<const uint4*>(o_seq + (int64_t)qpos * p.o_stride[2]) + chunk);
            if (chunk == 0) lv[ps] = __ldg(p.lse + stat_base + qpos);
          }
        }
      };
      auto stats_finish = [&](int n) {
        const int r = n % 3;
        mbar_wait(bars + BAR_Q_FULL + r, (n / 3) & 1);
        const uint8_t* sdo = ring_do(n);
        float* st = sStat + r * 2 * kTile;
#pragma unroll
        for (int ps = 0; ps < 8; ++ps) {
          const int rr = ps * 16 + rsub;
          const uint4 a = *reinterpret_cast<const uint4*>(sdo + swz_off<ROWB>(rr, chunk));
          const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, ow[4] = {ov[ps].x, ov[ps].y, ov[ps].z, ov[ps].w};
          float d = 0.f;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 fa = Elem<T>::unpack(aw[e]), fo = Elem<T>::unpack(ow[e]);
            d = fmaf(fa.x, fo.x, d);
            d = fmaf(fa.y, fo.y, d);
          }
          d += __shfl_xor_sync(0xffffffffu, d, 1);
          d += __shfl_xor_sync(0xffffffffu, d, 2);
          d += __shfl_xor_sync(0xffffffffu, d, 4);
          if (chunk == 0) {
            st[rr] = -lv[ps] * kLog2e;
            st[kTile + rr] = -d * p.scale;
          }
        }
        mbar_arrive_warp(bars + BAR_STAT + r);
      };

      if (g.cls && tid_g < kBlock) {
        sKpm0[tid_g] = p.kpm ? p.kpm[(int64_t)s.b * p.L + tid_g] * kLog2e : 0.f;
        sKpm0[kBlock + tid_g] = 0.f;
      }
      int stats_done = 0;
      for (; stats_done < 2 && stats_done < s.nqt; ++stats_done) {       // the first key tile starts on these
        stats_issue(stats_done);
        stats_finish(stats_done);
      }
      for (int j = 0; j < s.ntiles; ++j) {
        int kt, ub, ue;
        bool pre;
        g.tile(s, j, kt, pre, ub, ue);
        // the query tile the NEXT key tile starts to touch (two ahead of this tile's own): its O rows are requested now
        int want = (kt - s.t0) + 3;
        if (want > s.nqt) want = s.nqt;
        const int pending = stats_done < want ? stats_done : -1;
        if (pending >= 0) stats_issue(pending);

        mbar_wait(bars + BAR_ACC_READY, j & 1);
        mbar_wait(bars + BAR_ACC_READY2, j & 1);
        tc_fence_after();
        if (!pre) {
          const int n = kt - s.t0;
          uint8_t* stage[3] = {smem + S::OFF_K + (j & 1) * S::TILE, ring_do(n), ring_q(n)};        // dK, dV, dQ
          const uint32_t cols[3] = {(uint32_t)S::COL_DK, (uint32_t)S::COL_DV, (uint32_t)(S::COL_DQ + 64 * (kt & 1))};
#pragma unroll 1
          for (int which = 0; which < 3; ++which) {
#pragma unroll 1
            for (int half = 0; half < DH / 32; ++half) {
              uint32_t v[32];
              tmem_ld32(trow + cols[which] + 32 * half, v);
              tmem_wait_ld(v);
#pragma unroll
              for (int cq = 0; cq < 4; ++cq) {
                uint4 o;
                o.x = Elem<T>::pack(__uint_as_float(v[cq * 8 + 0]), __uint_as_float(v[cq * 8 + 1]));
                o.y = Elem<T>::pack(__uint_as_float(v[cq * 8 + 2]), __uint_as_float(v[cq * 8 + 3]));
                o.z = Elem<T>::pack(__uint_as_float(v[cq * 8 + 4]), __uint_as_float(v[cq * 8 + 5]));
                o.w = Elem<T>::pack(__uint_as_float(v[cq * 8 + 6]), __uint_as_float(v[cq * 8 + 7]));
                *reinterpret_cast<uint4*>(stage[which] + swz_off<ROWB>(row, half * 4 + cq)) = o;
              }
            }
            if (which == 1) {                 // dK and dV are out of TMEM: the next tile may start to accumulate
              tc_fence_before();
              mbar_arrive_warp(bars + BAR_ACC_FREE);
            }
          }
          fence_proxy_async();
          named_bar_sync(1, 128);
          if (tid_g == 0) {
            tma_store_4d(&tmDK, stage[0], 0, kt * kTile, s.h, s.b);
            tma_store_commit();
            tma_store_4d(&tmDV, stage[1], 0, kt * kTile, s.h, s.b);
            tma_store_4d(&tmDQ, stage[2], 0, kt * kTile, s.h, s.b);
            tma_store_commit();
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");      // the K buffer has been read
            mbar_arrive(bars + BAR_K_FREE + (j & 1));
            tma_store_wait_read();
            mbar_arrive(bars + BAR_RING_FREE + n % 3);
          }
        } else {                             // pre-tile: nothing to drain
          tc_fence_before();
          mbar_arrive_warp(bars + BAR_ACC_FREE);
          if (tid_g == 0) mbar_arrive(bars + BAR_K_FREE + (j & 1));
        }
        if (pending >= 0) {
          stats_finish(pending);
          ++stats_done;
        }
        for (; stats_done < want; ++stats_done) {      // (only if more than one query tile became due at once)
          stats_issue(stats_done);
          stats_finish(stats_done);
        }
      }
      if (g.cls) {
        // this segment's share of dK_0 / dV_0 -> fp32 partial [2 (dK, dV)][32 keys][DH]
        const int which = w < 2 ? 1 : 0;                 // lanes 0-63: dV_0^T (columns 0-31), lanes 64-127: dK_0^T (columns 32-63)
        const int d = (w & 1) * 32 + lane;
        uint32_t v[32];
        tmem_ld32(trow + S::COL_G + (which ? 0 : 32), v);
        tmem_wait_ld(v);
        float* dst = p.gpart + (((int64_t)s.seq * p.maxseg + s.gslot) * 2 + which) * (kBlock * DH) + d;
#pragma unroll
        for (int key = 0; key < kBlock; ++key) dst[key * DH] = __uint_as_float(v[key]);
      }
      if (tid_g == 0) tma_store_wait_all();
      segment_sync();
    }
  } else {
    // ================================================ math groups ==================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    const int wg = warp >> 2;
    const int c = warp & 3;                             // TMEM lane quarter = key block of the tile (band units)
    const int row = c * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(c * 32) << 16);
    uint8_t* sDS = smem + S::OFF_DS;
    uint8_t* sG = smem + S::OFF_G;

    for (int start = range_lo; start < range_hi;) {
      const B1Seg s = b1_make_seg(p, g, start, range_hi);
      start += s.t1 - s.t0;
      int u = 0, groups = 0, gtiles = 0, stat_waited = 0;
      for (int j = 0; j < s.ntiles; ++j) {
        int kt, ub, ue;
        bool pre;
        g.tile(s, j, kt, pre, ub, ue);
        const int kb = 4 * kt + c;
        const int kpos = kt * kTile + row;
        float kv = 0.f;                                 // additive mask of this lane's key (log2 domain)
        if (p.kpm && kpos < p.L) kv = p.kpm[(int64_t)s.b * p.L + kpos] * kLog2e;
        for (int pos = ub; pos < ue; ++pos, ++u) {
          const int slot = g.slot_of(pos);
          const bool last_x = slot == g.nx - 1, last_y = slot >= 4 && slot == g.nq - 1;
          const int grp = groups, gt = gtiles;
          if (last_x || last_y) ++groups;
          if (slot < 0) ++gtiles;
          if ((u & 1) != wg) continue;
          const int n = (kt - s.t0) + (slot < 0 ? 0 : (slot >> 2));
          for (; stat_waited <= n; ++stat_waited) mbar_wait(bars + BAR_STAT + stat_waited % 3, (stat_waited / 3) & 1);
          const float* st = sStat + (n % 3) * 2 * kTile;
          const uint32_t tb = trow + S::COL_U + 64 * wg;           // this group's score buffer
          const uint32_t ta = trow + S::COL_A + 32 * wg;           // ... and 16-bit operand buffer: P^T 0-15 | dS^T 16-31
          // the scores are pulled into registers and the buffer is handed back before the arithmetic starts
          auto release_scores = [&]() {
            tc_fence_before();
            mbar_arrive_warp(bars + BAR_U_FREE + wg);
          };
          auto wait_operands_free = [&]() {
            if (u >= 2) mbar_wait(bars + BAR_A_FREE + wg, ((u - 2) >> 1) & 1);
            tc_fence_after();
          };
          mbar_wait(bars + BAR_S_READY + wg, (u >> 1) & 1);
          tc_fence_after();
          // One code path for band units (lane = key of the tile, columns = the slot's 32 queries) and the global unit
          // (lane = query of the tile, columns = the 32 keys of block 0): x = S * scale*log2e + col_a[col] + row_a,
          // P = exp2(x), dS = P * (dP * scale + col_b[col] + row_b); the statistics -lse*log2e / -delta*scale are the
          // per-COLUMN terms of a band unit and the per-ROW terms of the global unit, the additive key mask the other way
          // round.  (One copy of the loop on purpose: the kernel is bound by instruction fetch as much as by any pipe.)
          uint32_t pk[16], dk[16];
          const bool is_g = slot < 0;
          const int qb = 4 * kt + (is_g ? c : slot);
          bool live;
          uint32_t keep = 0xffffffffu;                   // bit col clear: causally masked (diagonal blocks only)
          const float *col_a, *col_b;
          float row_a, row_b;
          if (!is_g) {
            live = kb < p.nb && qb < p.nb && slot >= c && slot <= c + p.left - 1 && !(g.cls && kb == 0);
            if (qb == kb) keep = 0xffffffffu << lane;     // key position > query position <=> lane > column
            col_a = st + (slot & 3) * kBlock;
            col_b = st + kTile + (slot & 3) * kBlock;
            row_a = kv;
            row_b = 0.f;
          } else {
            live = qb < p.nb;
            if (qb == 0) keep = lane == 31 ? 0xffffffffu : ((2u << lane) - 1u);      // key index > query index <=> column > lane
            col_a = sKpm0;
            col_b = sKpm0 + kBlock;                       // 32 zeros
            row_a = st[row];
            row_b = st[kTile + row];
          }
          if (live) {
            uint32_t sv[32], dv[32];
            tmem_ld32(tb, sv);
            tmem_ld32(tb + 32, dv);
            tmem_wait_ld(sv, dv);
            release_scores();
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
              const float4 a4 = reinterpret_cast<const float4*>(col_a)[c4], b4 = reinterpret_cast<const float4*>(col_b)[c4];
              const float ca[4] = {a4.x, a4.y, a4.z, a4.w}, cb[4] = {b4.x, b4.y, b4.z, b4.w};
              float pp[4], dd[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int col = c4 * 4 + e;
                float pe = fast_exp2(fmaf(__uint_as_float(sv[col]), p.scale_log2, ca[e]) + row_a);
                if (!((keep >> col) & 1u)) pe = 0.f;
                pp[e] = pe;
                dd[e] = pe * (fmaf(__uint_as_float(dv[col]), p.scale, cb[e]) + row_b);
              }
              pk[c4 * 2] = Elem<T>::pack(pp[0], pp[1]);
              pk[c4 * 2 + 1] = Elem<T>::pack(pp[2], pp[3]);
              dk[c4 * 2] = Elem<T>::pack(dd[0], dd[1]);
              dk[c4 * 2 + 1] = Elem<T>::pack(dd[2], dd[3]);
            }
          } else {
            release_scores();
#pragma unroll
            for (int e = 0; e < 16; ++e) pk[e] = dk[e] = 0u;
          }
          wait_operands_free();
          if (!is_g) {
            tmem_st16(ta, pk);
            tmem_st16(ta + 16, dk);
            // dS^T row of this key -> staging tile (the dQ MMAs of the previous group must have read it)
            if (grp >= 1) mbar_wait(bars + BAR_DS_FREE, (grp - 1) & 1);
            uint8_t* half = sDS + ((slot & 3) >> 1) * S::TILE;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
              *reinterpret_cast<uint4*>(half + swz_off<128>(row, (slot & 1) * 4 + ch)) =
                  make_uint4(dk[4 * ch], dk[4 * ch + 1], dk[4 * ch + 2], dk[4 * ch + 3]);
            if (last_y) {                               // slots of the group that do not exist contribute nothing
              for (int sp = (slot & 3) + 1; sp < 4; ++sp) {
                uint8_t* hz = sDS + (sp >> 1) * S::TILE;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch)
                  *reinterpret_cast<uint4*>(hz + swz_off<128>(row, (sp & 1) * 4 + ch)) = make_uint4(0, 0, 0, 0);
              }
            }
          } else {
            tmem_st16(ta, dk);                          // A operand of dQ X += dS_g K_0
            if (gt >= 1) mbar_wait(bars + BAR_G_FREE, (gt - 1) & 1);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {            // row of [P_g (64 B) | dS_g (64 B)]
              *reinterpret_cast<uint4*>(sG + swz_off<128>(row, ch)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
              *reinterpret_cast<uint4*>(sG + swz_off<128>(row, 4 + ch)) = make_uint4(dk[4 * ch], dk[4 * ch + 1], dk[4 * ch + 2], dk[4 * ch + 3]);
            }
          }
          fence_proxy_async();                          // staging tiles are read by the tensor core (async proxy)
          tmem_wait_st();
          tc_fence_before();
          mbar_arrive_warp(bars + BAR_P_READY + wg);
          if (slot >= 0) mbar_arrive_warp(bars + (slot < 4 ? BAR_GRPX_READY : BAR_GRPY_READY));
        }
      }
      segment_sync();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 15) tmem_dealloc<512>(tmem_base);
}

// dK / dV rows of the global key block: sum of the sequence's per-segment partials in segment order.
template <typename T, int DH>
__global__ void __launch_bounds__(256) attn_bwd_finish_kernel(const B1Params p, T* __restrict__ dk, T* __restrict__ dv,
                                                              int64_t dk_sb, int64_t dk_sh, int64_t dk_sr, int64_t dv_sb,
                                                              int64_t dv_sh, int64_t dv_sr) {
  // grid (2 * 32 * DH / 256, B*H): one output element per thread, the partials of a sequence are read in parallel
  const int seq = blockIdx.y, b = seq / p.H, h = seq % p.H;
  const int first = b1_cta_of(seq * p.T, p.num_tiles, p.num_ctas), last = b1_cta_of(seq * p.T + p.T - 1, p.num_tiles, p.num_ctas);
  const int nseg = last - first + 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int which = i / (kBlock * DH), e = i % (kBlock * DH), key = e / DH, d = e % DH;
  const float* src = p.gpart + (((int64_t)seq * p.maxseg) * 2 + which) * (kBlock * DH) + e;
  float part[8];
  float acc = 0.f;
  for (int k0 = 0; k0 < nseg; k0 += 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) part[k] = (k0 + k < nseg) ? __ldcg(src + (int64_t)(k0 + k) * 2 * (kBlock * DH)) : 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc += part[k];          // fixed order: segment 0, 1, 2, ...
  }
  if (which == 0) dk[b * dk_sb + h * dk_sh + key * dk_sr + d] = from_f32<T>(acc);
  else dv[b * dv_sb + h * dv_sh + key * dv_sr + d] = from_f32<T>(acc);
}

// ------------------------------------------------------------------------------------------ host side
static int b1_num_ctas(int num_tiles) {
  const int sms = sm_count_of_current_device();
  return num_tiles < sms ? num_tiles : sms;
}

static int b1_maxseg(int BH, int T, int num_tiles, int num_ctas) {
  int m = 1;
  for (int s = 0; s < BH; ++s) {
    const int n = b1_cta_of(s * T + T - 1, num_tiles, num_ctas) - b1_cta_of(s * T, num_tiles, num_ctas) + 1;
    if (n > m) m = n;
  }
  return m;
}

bool bwd1_supported(const svae_attn_desc* d) {
  if (d->dtype != SVAE_DTYPE_BF16 && d->dtype != SVAE_DTYPE_F16) return false;
  if (d->head_dim != 64 || !(d->scale > 0.f) || !d->causal) return false;
  const Band b = make_band(d->window_size, d->causal, d->include_cls);
  return b.nsup == 0 && b.left >= 1 && b.left <= kB1MaxLeft;
}

static size_t b1_align256(size_t x) { return (x + 255) & ~size_t(255); }

size_t bwd1_workspace(const svae_attn_desc* d) {
  if (!d->include_cls) return 256;
  const int T = (d->seq_len + kTile - 1) / kTile, BH = d->batch * d->heads;
  const int num_tiles = BH * T, num_ctas = b1_num_ctas(num_tiles);
  return b1_align256(sizeof(float) * (size_t)BH * b1_maxseg(BH, T, num_tiles, num_ctas) * 2 * kBlock * d->head_dim);
}

template <typename T, int DH>
static int launch_bwd1(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out,
                       const void* dout, const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace,
                       cudaStream_t st) {
  using S = B1Smem<DH>;
  const int B = d->batch, H = d->heads, L = d->seq_len;
  const Band band = make_band(d->window_size, d->causal, d->include_cls);
  B1Params p;
  p.kpm = kpm; p.lse = lse; p.out = out;
  p.o_stride[0] = d->o_stride[0]; p.o_stride[1] = d->o_stride[1]; p.o_stride[2] = d->o_stride[2];
  p.gpart = reinterpret_cast<float*>(workspace);
  p.L = L; p.H = H; p.T = (L + kTile - 1) / kTile; p.nb = L / kBlock;
  p.left = band.left; p.cls = band.cls; p.nq = band.left + 3;
  p.num_tiles = B * H * p.T;
  p.num_ctas = b1_num_ctas(p.num_tiles);
  p.maxseg = band.cls ? b1_maxseg(B * H, p.T, p.num_tiles, p.num_ctas) : 1;
  p.scale = d->scale; p.scale_log2 = d->scale * kLog2e;

  const CUtensorMapDataType dt = Elem<T>::tm;
  CUtensorMap tQ, tDO, tK, tV, tK32, tV32, tDQ, tDK, tDV;
  int rc;
#define SVAE_TM(map, ptr, strd, rows) \
  if ((rc = encode_tmap(&map, dt, ptr, DH, L, H, B, strd, rows))) return rc
  SVAE_TM(tQ, q, d->q_stride, kTile);     SVAE_TM(tDO, dout, d->do_stride, kTile);
  SVAE_TM(tK, k, d->k_stride, kTile);     SVAE_TM(tV, v, d->v_stride, kTile);
  SVAE_TM(tK32, k, d->k_stride, kBlock);  SVAE_TM(tV32, v, d->v_stride, kBlock);
  SVAE_TM(tDQ, dq, d->dq_stride, kTile);  SVAE_TM(tDK, dk, d->dk_stride, kTile);
  SVAE_TM(tDV, dv, d->dv_stride, kTile);
#undef SVAE_TM

  auto kern = attn_bwd1_sm100_kernel<T, DH>;
  SVAE_CONFIGURE_SMEM(kern, S::DYN_BYTES);
  {
    ScopedKernelTimer timer("attn_bwd_sm100", st);
    kern<<<p.num_ctas, kB1Threads, S::DYN_BYTES, st>>>(tQ, tDO, tK, tV, tK32, tV32, tDQ, tDK, tDV, p);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  if (band.cls) {
    ScopedKernelTimer timer("attn_bwd_finish", st);
    attn_bwd_finish_kernel<T, DH><<<dim3(2 * kBlock * DH / 256, B * H), 256, 0, st>>>(p, reinterpret_cast<T*>(dk), reinterpret_cast<T*>(dv), d->dk_stride[0],
                                                         d->dk_stride[1], d->dk_stride[2], d->dv_stride[0], d->dv_stride[1],
                                                         d->dv_stride[2]);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  return SVAE_OK;
}

int bwd1(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out, const void* dout,
         const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace, cudaStream_t st) {
  if (d->dtype == SVAE_DTYPE_BF16) return launch_bwd1<__nv_bfloat16, 64>(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
  return launch_bwd1<__half, 64>(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
}

}  // namespace sm100
}  // namespace svae
