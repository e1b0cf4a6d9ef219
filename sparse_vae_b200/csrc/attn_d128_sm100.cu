// Block-sparse CAUSAL attention at head size 128 for sm_100a (tcgen05 / TMEM / TMA): the attention of sparse decoders
// of width 1024 (the layout has 8 heads whatever the width, so d_model 1024 means heads of 128).
//
// The head-64 kernels hold a query tile's whole band in shared memory and TMEM at once.  At head 128 that does not fit
// (window 10 with the global block: 14 slots of 32 keys = 2 x 112 KB of K / V, 448 + 128 TMEM columns), so every pass
// here streams the key (or query) side in GROUPS of four 32-row slots = 128 rows, with the structure of
// causal_attn_sm100.cu: 6 warps, warps 0-3 math (one TMEM lane quarter = one 32-row block each, so block sparsity is
// warp-uniform), warp 4 TMA, warp 5 MMA issue.
//
// Operand layout (attn_sm100.cuh, kmajor_desc / mnmajor_desc): every 128-row operand tile arrives as two TMA boxes of
// 64 columns, stored as two 16 KB halves.
//
// Forward (one CTA per 128-query tile): the tile's key slots (global block 0 when include_cls, then the band
// 4t-(left-1) .. 4t+3) are streamed four at a time through a 2-stage TMA ring; S = Q K^T double-buffered in TMEM
// (2 x 128 columns), online softmax over the groups with lazy rescaling of O (128 columns), P written over S as
// 16-bit, O += P V.  Slots that are dead for a warp's block-row get P = 0.  Shared memory 160 KB.
//
// Backward: three launches, no atomics, bit-deterministic.
//   dQ pass     one CTA per query tile over the same slot groups: Q, dO resident; S = Q K^T and dP = dO V^T
//               (128 x 128 each) into TMEM, dS = P o (dP - delta) * scale written over S as 16-bit, dQ += dS K.
//               delta = rowsum(dO o O) is computed here for the second pass.  With include_cls the tile also forms
//               its share of key block 0's gradients: [P_0 | dS_0] (128 queries x 64) is staged in shared memory and
//               dV_0^T += dO^T [P_0 | dS_0], dK_0^T += Q^T [P_0 | dS_0] (columns 0-31 resp. 32-63 are used), written
//               as one fp32 partial per query tile.
//   dK/dV pass  one CTA per key tile kt: K, V resident; query tiles kt .. kt + ceil((left+3)/4) - 1 streamed.
//               S^T = K Q^T, dP^T = V dO^T, P^T and dS^T over them as 16-bit, dV += P^T dO, dK += dS^T Q.  Key block 0
//               is skipped when include_cls (every query attends it: its rows come from the partials).
//   finish      dK / dV rows of key block 0: the partials of a sequence summed in query-tile order.
// TMEM: forward S 0 / 128, O 256; dQ pass S 0, dP 128, dQ 256, dV_0^T 384, dK_0^T 448; dK/dV pass S^T 0, dP^T 128,
// dV 256, dK 384.
#include <type_traits>

#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kDThreads = 192;          // warps 0-3: math (one TMEM lane quarter each), 4: TMA, 5: MMA issue
constexpr int kDH = 128;
constexpr int kDHalf = kTile * 128;     // one 64-column half of a 128-row tile: 16 KB
constexpr int kDTileB = 2 * kDHalf;     // a 128-row x 128-column 16-bit tile: 32 KB
constexpr int kDMaxLeft = 10;           // windows 1..10: at most 14 key slots per query tile
constexpr float kDRescale = 8.0f;       // log2 units the running maximum may lag behind before O is rescaled

struct DFwdSmem {
  static constexpr int OFF_Q = 0;                                 // later the output staging tile
  static constexpr int OFF_K = OFF_Q + kDTileB;                   // [2] slot groups
  static constexpr int OFF_V = OFF_K + 2 * kDTileB;               // [2]
  static constexpr int OFF_KPM = OFF_V + 2 * kDTileB;             // [2][128] additive key terms (log2 domain)
  static constexpr int OFF_BAR = OFF_KPM + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
};

struct DDqSmem {
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_DO = OFF_Q + kDTileB;
  static constexpr int OFF_K = OFF_DO + kDTileB;                  // [2]
  static constexpr int OFF_V = OFF_K + 2 * kDTileB;               // [2]
  static constexpr int OFF_G = OFF_V + 2 * kDTileB;               // [128 queries][P_0 (32 keys) | dS_0 (32 keys)]
  static constexpr int OFF_KPM = OFF_G + kDHalf;                  // [2][128]
  static constexpr int OFF_BAR = OFF_KPM + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int COL_S = 0, COL_DP = 128, COL_DQ = 256, COL_GV = 384, COL_GK = 448;
  static_assert(DYN_BYTES <= 227 * 1024, "shared memory");
};

struct DKvSmem {
  static constexpr int OFF_K = 0;
  static constexpr int OFF_V = OFF_K + kDTileB;
  static constexpr int OFF_Q = OFF_V + kDTileB;                   // [2] query tiles
  static constexpr int OFF_DO = OFF_Q + 2 * kDTileB;              // [2]
  static constexpr int OFF_STAT = OFF_DO + 2 * kDTileB;           // [2][-lse*log2e (128) | -delta*scale (128)]
  static constexpr int OFF_BAR = OFF_STAT + 4 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int COL_S = 0, COL_DP = 128, COL_DV = 256, COL_DK = 384;
  static_assert(DYN_BYTES <= 227 * 1024, "shared memory");
};

struct DParams {
  const float* kpm;     // [B, L] additive or null
  float* lse;           // [B, H, L] natural log (written by the forward, read by the backward)
  float* delta;         // [B, H, L] rowsum(dO o O): dQ pass -> dK/dV pass
  float* gpart;         // [B*H][T][2 (dK, dV)][32 keys][128] fp32 partials of key block 0
  const void *out, *dout;
  void *dq, *dk, *dv;
  int64_t o_stride[3], do_stride[3], dq_stride[3], dk_stride[3], dv_stride[3];
  int L, H, T, nb;      // T = 128-row tiles, nb = 32-row blocks
  int left, cls;        // band width (sub-diagonals incl. the main one), global block 0
  int ns, ng;           // key slots of a query tile, groups of four slots
  float scale, scale_log2;
};

// key block of slot j of query tile t (slot 0 = block 0 when cls, then the band)
__device__ __forceinline__ int d_slot_block(const DParams& p, int t, int j) {
  return (p.cls && j == 0) ? 0 : 4 * t - (p.left - 1) + j - p.cls;
}
// the slot carries keys of the sequence that are not a duplicate of the global block
__device__ __forceinline__ bool d_slot_valid(const DParams& p, int t, int j) {
  if (j >= p.ns) return false;
  if (p.cls && j == 0) return true;
  const int blk = d_slot_block(p, t, j);
  return blk >= p.cls && blk < p.nb;
}
// block-row r attends the slot
__device__ __forceinline__ bool d_slot_live(const DParams& p, int t, int j, int r) {
  if (r >= p.nb || !d_slot_valid(p, t, j)) return false;
  if (p.cls && j == 0) return true;
  const int blk = d_slot_block(p, t, j);
  return blk >= r - (p.left - 1) && blk <= r;
}
__device__ __forceinline__ float d_key_term(const DParams& p, int b, int key) {
  if (key >= p.L) return -INFINITY;
  return p.kpm ? p.kpm[(int64_t)b * p.L + key] * kLog2e : 0.f;
}

// 128-row x 128-column tile -> two TMA boxes of 64 columns
__device__ __forceinline__ void d_load_tile(uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int row, int h, int b) {
  load_rows<kDH>(dst, kDHalf, map, bar, row, h, b);
}

// 128 fp32 TMEM columns of one row -> 16-bit -> global row (16-byte stores)
template <typename T>
__device__ __forceinline__ void d_store_row(uint32_t taddr, T* dst, bool ok) {
#pragma unroll 1
  for (int qq = 0; qq < 4; ++qq) {
    uint32_t v[32];
    tmem_ld32(taddr + 32 * qq, v);
    tmem_wait_ld(v);
    if (ok) {
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        uint4 o;
        o.x = Elem<T>::pack(__uint_as_float(v[cq * 8 + 0]), __uint_as_float(v[cq * 8 + 1]));
        o.y = Elem<T>::pack(__uint_as_float(v[cq * 8 + 2]), __uint_as_float(v[cq * 8 + 3]));
        o.z = Elem<T>::pack(__uint_as_float(v[cq * 8 + 4]), __uint_as_float(v[cq * 8 + 5]));
        o.w = Elem<T>::pack(__uint_as_float(v[cq * 8 + 6]), __uint_as_float(v[cq * 8 + 7]));
        reinterpret_cast<uint4*>(dst)[qq * 4 + cq] = o;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ forward
template <typename T>
__global__ void __launch_bounds__(kDThreads, 1)
attn_d128_fwd_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                           const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const DParams p) {
  using S = DFwdSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;                 // [2]
  uint64_t* v_full = bars + 3;                 // [2]
  uint64_t* kv_free = bars + 5;                // [2] both MMAs that read the stage have retired
  uint64_t* s_ready = bars + 7;                // [2]
  uint64_t* p_ready = bars + 9;                // [2] (128 arrivals)
  uint64_t* o_done = bars + 11;                // P V of a group retired
  uint64_t* o_final = bars + 12;               // every MMA of the CTA retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int ng = p.ng;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(k_full + s, 1); mbar_init(v_full + s, 1); mbar_init(kv_free + s, 1);
      mbar_init(s_ready + s, 1); mbar_init(p_ready + s, 128);
    }
    mbar_init(o_done, 1);
    mbar_init(o_final, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    if (lane == 0) { prefetch_tensormap(&tmQ); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV); prefetch_tensormap(&tmO); }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t COL_O = 256;

  if (warp == 4) {
    // ---- TMA producer: Q, then per group four K slots and four V slots (rows outside [0, L) arrive as zeros)
    mbar_arrive_expect_tx_w(q_full, kDTileB);
    d_load_tile(smem + S::OFF_Q, &tmQ, q_full, t * kTile, h, b);
    for (int i = 0; i < ng; ++i) {
      const int s = i & 1;
      if (i >= 2) mbar_wait(kv_free + s, ((i >> 1) - 1) & 1);
      uint8_t* kd = smem + S::OFF_K + s * kDTileB;
      uint8_t* vd = smem + S::OFF_V + s * kDTileB;
      mbar_arrive_expect_tx_w(k_full + s, kDTileB);
      for (int c = 0; c < 4; ++c) {
        const int row = d_slot_block(p, t, 4 * i + c) * kBlock;
        tma_load_4d_w(kd + c * kBlock * 128, &tmK, k_full + s, 0, row, h, b);
        tma_load_4d_w(kd + kDHalf + c * kBlock * 128, &tmK, k_full + s, 64, row, h, b);
      }
      mbar_arrive_expect_tx_w(v_full + s, kDTileB);
      for (int c = 0; c < 4; ++c) {
        const int row = d_slot_block(p, t, 4 * i + c) * kBlock;
        tma_load_4d_w(vd + c * kBlock * 128, &tmV, v_full + s, 0, row, h, b);
        tma_load_4d_w(vd + kDHalf + c * kBlock * 128, &tmV, v_full + s, 64, row, h, b);
      }
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S(0); then per group  S(i+1) ; wait P(i) ; O += P(i) V(i)   (in-order pipe: S(i+1) overwrites the
    //      buffer of P(i-1) only after P(i-1) V(i-1) has read it)
    const uint32_t idesc_s = make_idesc(kTile, kTile, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_pv = make_idesc(kTile, kDH, Elem<T>::fmt, 0, 1);
    const uint32_t q_addr = smem_u32(smem + S::OFF_Q);
    auto issue_s = [&](int i) {
      const int s = i & 1;
      mbar_wait(k_full + s, (i >> 1) & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * kDTileB);
#pragma unroll
      for (int ks = 0; ks < kDH / 16; ++ks)
        mma_ss_w(tmem_base + 128 * s, kmajor_desc(q_addr, ks, kDHalf), kmajor_desc(k_addr, ks, kDHalf), idesc_s, ks > 0 ? 1u : 0u);
      tc_commit_w(s_ready + s);
    };
    mbar_wait(q_full, 0);
    issue_s(0);
    for (int i = 0; i < ng; ++i) {
      if (i + 1 < ng) issue_s(i + 1);
      const int s = i & 1;
      mbar_wait(p_ready + s, (i >> 1) & 1);
      mbar_wait(v_full + s, (i >> 1) & 1);
      tc_fence_after();
      const uint32_t v_addr = smem_u32(smem + S::OFF_V + s * kDTileB);
#pragma unroll
      for (int k2 = 0; k2 < kTile / 16; ++k2)           // 16 keys per MMA: A = P (16-bit, 8 columns), B = V MN-major
        mma_ts_w(tmem_base + COL_O, tmem_base + 128 * s + 8 * k2, mnmajor_desc(v_addr, k2, kDHalf), idesc_pv, (i > 0 || k2 > 0) ? 1u : 0u);
      tc_commit_w(o_done);
      tc_commit_w(kv_free + s);
    }
    tc_commit_w(o_final);
  } else {
    // ---- softmax / epilogue warps: warp w owns block-row r = 4t + w = TMEM lanes 32w ..
    const int row = warp * 32 + lane;
    const int r = 4 * t + warp;
    const int qpos = t * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    float m = -INFINITY, l = 0.f;                        // running maximum (log2 domain) and row sum relative to it
    for (int i = 0; i < ng; ++i) {
      float* kp = sKpm + (i & 1) * kTile;
      {
        const int j = 4 * i + (int)(threadIdx.x >> 5);
        float kv = 0.f;
        if (p.kpm && d_slot_valid(p, t, j)) kv = p.kpm[(int64_t)b * p.L + d_slot_block(p, t, j) * kBlock + lane] * kLog2e;
        kp[threadIdx.x] = kv;
      }
      named_bar_sync(1, 128);
      mbar_wait(s_ready + (i & 1), (i >> 1) & 1);
      tc_fence_after();
      const uint32_t ts = trow + 128 * (i & 1);
      // pass 1: maximum over the live slots of the group (warp-uniform liveness; the diagonal block masks keys > row)
      float tmax = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int j = 4 * i + c;
        if (!d_slot_live(p, t, j, r)) continue;
        const bool diag = d_slot_block(p, t, j) == r;
        uint32_t v[32];
        tmem_ld32(ts + 32 * c, v);
        tmem_wait_ld(v);
        const float4* k4 = reinterpret_cast<const float4*>(kp + 32 * c);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float4 kk = k4[e];
          const float kx[4] = {kk.x, kk.y, kk.z, kk.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float x = fmaf(__uint_as_float(v[4 * e + u]), p.scale_log2, kx[u]);
            if (diag && 4 * e + u > lane) x = -INFINITY;
            tmax = fmaxf(tmax, x);
          }
        }
      }
      float alpha = 1.f;
      if (tmax > m + kDRescale || m == -INFINITY) {      // (also the first group)
        alpha = (m == -INFINITY) ? 0.f : fast_exp2(m - tmax);
        m = tmax;
        l *= alpha;
      }
      const float neg_m = (m == -INFINITY) ? 0.f : -m;
      // pass 2: P = exp2(s * scale*log2e + mask - m) written over S as 16-bit, left to right; dead slots P = 0
      float l0 = 0.f, l1 = 0.f;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int j = 4 * i + c;
        uint32_t pk[16];
        if (d_slot_live(p, t, j, r)) {
          const bool diag = d_slot_block(p, t, j) == r;
          uint32_t v[32];
          tmem_ld32(ts + 32 * c, v);
          tmem_wait_ld(v);
          const float4* k4 = reinterpret_cast<const float4*>(kp + 32 * c);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float4 kk = k4[e];
            const float kx[4] = {kk.x, kk.y, kk.z, kk.w};
            float pe[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              pe[u] = fast_exp2(fmaf(__uint_as_float(v[4 * e + u]), p.scale_log2, kx[u]) + neg_m);
              if (diag && 4 * e + u > lane) pe[u] = 0.f;
            }
            l0 += pe[0] + pe[2];
            l1 += pe[1] + pe[3];
            pk[2 * e] = Elem<T>::pack(pe[0], pe[1]);
            pk[2 * e + 1] = Elem<T>::pack(pe[2], pe[3]);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) pk[e] = 0u;
        }
        tmem_st16(ts + 16 * c, pk);
      }
      l += l0 + l1;
      // lazy rescaling of the accumulator: O holds sums relative to the OLD maximum
      const bool any = __any_sync(0xffffffffu, alpha != 1.f);
      if (any && i > 0) {
        mbar_wait(o_done, (i - 1) & 1);                  // P V of the previous group has retired
        tc_fence_after();
#pragma unroll 1
        for (int qq = 0; qq < kDH / 32; ++qq) {
          uint32_t o[32];
          tmem_ld32(trow + COL_O + 32 * qq, o);
          tmem_wait_ld(o);
#pragma unroll
          for (int e = 0; e < 32; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
          uint32_t lo[16], hi[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) { lo[e] = o[e]; hi[e] = o[16 + e]; }
          tmem_st16(trow + COL_O + 32 * qq, lo);
          tmem_st16(trow + COL_O + 32 * qq + 16, hi);
        }
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_ready + (i & 1));
    }
    // epilogue: O / l -> 16-bit -> swizzled staging (the Q tile, two halves) -> TMA store ; LSE
    mbar_wait(o_final, 0);
    tc_fence_after();
    uint8_t* stage = smem + S::OFF_Q;
    const float inv = 1.0f / l;                          // l == 0 (row with every key masked) -> NaN, like the reference
#pragma unroll 1
    for (int qq = 0; qq < kDH / 32; ++qq) {
      uint32_t o[32];
      tmem_ld32(trow + COL_O + 32 * qq, o);
      tmem_wait_ld(o);
      uint8_t* half = stage + (qq >> 1) * kDHalf;
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        uint4 w4;
        w4.x = Elem<T>::pack(__uint_as_float(o[cq * 8 + 0]) * inv, __uint_as_float(o[cq * 8 + 1]) * inv);
        w4.y = Elem<T>::pack(__uint_as_float(o[cq * 8 + 2]) * inv, __uint_as_float(o[cq * 8 + 3]) * inv);
        w4.z = Elem<T>::pack(__uint_as_float(o[cq * 8 + 4]) * inv, __uint_as_float(o[cq * 8 + 5]) * inv);
        w4.w = Elem<T>::pack(__uint_as_float(o[cq * 8 + 6]) * inv, __uint_as_float(o[cq * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(half + swz_off<128>(row, (qq & 1) * 4 + cq)) = w4;
      }
    }
    if (qpos < p.L) p.lse[((int64_t)b * p.H + h) * p.L + qpos] = (m + log2f(l)) * kLn2;
    fence_proxy_async();
    named_bar_sync(1, 128);
    if (threadIdx.x == 0) {
      tma_store_4d(&tmO, stage, 0, t * kTile, h, b);     // rows >= L are outside the tensor: clipped
      tma_store_4d(&tmO, stage + kDHalf, 64, t * kTile, h, b);
      tma_store_commit();
      tma_store_wait_all();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------ dQ pass
template <typename T>
__global__ void __launch_bounds__(kDThreads, 1)
attn_d128_bwd_dq_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                              const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV, const DParams p) {
  using S = DDqSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;                 // Q and dO
  uint64_t* kv_full = bars + 1;                // [2] K and V slot group
  uint64_t* kv_free = bars + 3;                // [2] the MMAs that read the stage have retired
  uint64_t* s_ready = bars + 5;                // S and dP of a group are in TMEM
  uint64_t* ds_ready = bars + 6;               // dS of a group is in TMEM (and [P_0 | dS_0] in shared memory), 128 arrivals
  uint64_t* dq_done = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int ng = p.ng;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(kv_full + s, 1); mbar_init(kv_free + s, 1); }
    mbar_init(s_ready, 1); mbar_init(ds_ready, 128); mbar_init(dq_done, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    if (lane == 0) { prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV); }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ---- TMA producer
    mbar_arrive_expect_tx_w(q_full, 2 * kDTileB);
    d_load_tile(smem + S::OFF_Q, &tmQ, q_full, t * kTile, h, b);
    d_load_tile(smem + S::OFF_DO, &tmDO, q_full, t * kTile, h, b);
    for (int i = 0; i < ng; ++i) {
      const int s = i & 1;
      if (i >= 2) mbar_wait(kv_free + s, ((i >> 1) - 1) & 1);
      uint8_t* kd = smem + S::OFF_K + s * kDTileB;
      uint8_t* vd = smem + S::OFF_V + s * kDTileB;
      mbar_arrive_expect_tx_w(kv_full + s, 2 * kDTileB);
      for (int c = 0; c < 4; ++c) {
        const int row = d_slot_block(p, t, 4 * i + c) * kBlock;
        tma_load_4d_w(kd + c * kBlock * 128, &tmK, kv_full + s, 0, row, h, b);
        tma_load_4d_w(kd + kDHalf + c * kBlock * 128, &tmK, kv_full + s, 64, row, h, b);
        tma_load_4d_w(vd + c * kBlock * 128, &tmV, kv_full + s, 0, row, h, b);
        tma_load_4d_w(vd + kDHalf + c * kBlock * 128, &tmV, kv_full + s, 64, row, h, b);
      }
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S, dP of group i ; wait dS(i) ; dQ += dS(i) K(i) (+ key block 0's products) ; S, dP of group i+1
    //      (in-order pipe: they overwrite dS(i) only after the dQ MMAs have read it)
    const uint32_t idesc_s = make_idesc(kTile, kTile, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_dq = make_idesc(kTile, kDH, Elem<T>::fmt, 0, 1);
    const uint32_t idesc_g = make_idesc(kTile, 64, Elem<T>::fmt, 1, 1);      // A and B MN-major, N = 64
    const uint32_t q_addr = smem_u32(smem + S::OFF_Q), do_addr = smem_u32(smem + S::OFF_DO);
    const uint32_t g_addr = smem_u32(smem + S::OFF_G);
    auto issue_sdp = [&](int i) {
      const int s = i & 1;
      mbar_wait(kv_full + s, (i >> 1) & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * kDTileB), v_addr = smem_u32(smem + S::OFF_V + s * kDTileB);
#pragma unroll
      for (int ks = 0; ks < kDH / 16; ++ks) {
        mma_ss_w(tmem_base + S::COL_S, kmajor_desc(q_addr, ks, kDHalf), kmajor_desc(k_addr, ks, kDHalf), idesc_s, ks > 0 ? 1u : 0u);
        mma_ss_w(tmem_base + S::COL_DP, kmajor_desc(do_addr, ks, kDHalf), kmajor_desc(v_addr, ks, kDHalf), idesc_s, ks > 0 ? 1u : 0u);
      }
      tc_commit_w(s_ready);
    };
    mbar_wait(q_full, 0);
    issue_sdp(0);
    for (int i = 0; i < ng; ++i) {
      const int s = i & 1;
      mbar_wait(ds_ready, i & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * kDTileB);
#pragma unroll
      for (int k2 = 0; k2 < kTile / 16; ++k2)          // 16 keys per MMA: A = dS (16-bit, 8 columns), B = K MN-major
        mma_ts_w(tmem_base + S::COL_DQ, tmem_base + S::COL_S + 8 * k2, mnmajor_desc(k_addr, k2, kDHalf), idesc_dq, (i > 0 || k2 > 0) ? 1u : 0u);
      if (p.cls && i == 0) {
        // dV_0^T (+)= dO^T [P_0 | dS_0], dK_0^T (+)= Q^T [P_0 | dS_0]: M = 128 head columns (two halves, MN-major),
        // K = 128 queries, N = 64
#pragma unroll
        for (int k2 = 0; k2 < kTile / 16; ++k2) {
          const uint64_t bd = make_smem_desc(g_addr + k2 * 16 * 128, 16 * 128, 1024, 128);
          mma_ss_w(tmem_base + S::COL_GV, make_smem_desc(do_addr + k2 * 16 * 128, kDHalf, 1024, 128), bd, idesc_g, k2 > 0 ? 1u : 0u);
          mma_ss_w(tmem_base + S::COL_GK, make_smem_desc(q_addr + k2 * 16 * 128, kDHalf, 1024, 128), bd, idesc_g, k2 > 0 ? 1u : 0u);
        }
      }
      tc_commit_w(kv_free + s);
      if (i + 1 < ng) issue_sdp(i + 1);
      else tc_commit_w(dq_done);
    }
  } else {
    // ---- math warps: warp w owns block-row r = 4t + w
    const int row = warp * 32 + lane;
    const int r = 4 * t + warp;
    const int qpos = t * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    const int64_t stat_idx = ((int64_t)b * p.H + h) * p.L + qpos;
    // delta = rowsum(dO o O) straight from global memory; rows >= L (zero Q and dO) get neutral statistics
    float nl = 0.f, nd = 0.f;
    if (qpos < p.L) {
      const T* o = reinterpret_cast<const T*>(p.out) + b * p.o_stride[0] + h * p.o_stride[1] + (int64_t)qpos * p.o_stride[2];
      const T* d_o = reinterpret_cast<const T*>(p.dout) + b * p.do_stride[0] + h * p.do_stride[1] + (int64_t)qpos * p.do_stride[2];
      float d = 0.f;
#pragma unroll 4
      for (int ch = 0; ch < kDH / 8; ++ch) {
        const uint4 a = reinterpret_cast<const uint4*>(o)[ch], g = reinterpret_cast<const uint4*>(d_o)[ch];
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 fa = Elem<T>::unpack(aw[e]), fg = Elem<T>::unpack(gw[e]);
          d = fmaf(fa.x, fg.x, d);
          d = fmaf(fa.y, fg.y, d);
        }
      }
      p.delta[stat_idx] = d;
      nl = -p.lse[stat_idx] * kLog2e;
      nd = -d * p.scale;
    }
    uint8_t* sG = smem + S::OFF_G;
    for (int i = 0; i < ng; ++i) {
      float* kp = sKpm + (i & 1) * kTile;
      {
        const int j = 4 * i + (int)(threadIdx.x >> 5);
        float kv = 0.f;
        if (p.kpm && d_slot_valid(p, t, j)) kv = p.kpm[(int64_t)b * p.L + d_slot_block(p, t, j) * kBlock + lane] * kLog2e;
        kp[threadIdx.x] = kv;
      }
      named_bar_sync(1, 128);
      mbar_wait(s_ready, i & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int j = 4 * i + c;
        uint32_t pk[16], dsk[16];
        if (d_slot_live(p, t, j, r)) {
          const bool diag = d_slot_block(p, t, j) == r;
          uint32_t sv[32], dv[32];
          tmem_ld32(trow + S::COL_S + 32 * c, sv);
          tmem_ld32(trow + S::COL_DP + 32 * c, dv);
          tmem_wait_ld(sv, dv);
          const float* kc = kp + 32 * c;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float pe[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              pe[u] = fast_exp2(fmaf(__uint_as_float(sv[e + u]), p.scale_log2, kc[e + u]) + nl);
              if (diag && e + u > lane) pe[u] = 0.f;
            }
            const float d0 = pe[0] * fmaf(__uint_as_float(dv[e]), p.scale, nd);
            const float d1 = pe[1] * fmaf(__uint_as_float(dv[e + 1]), p.scale, nd);
            pk[e >> 1] = Elem<T>::pack(pe[0], pe[1]);
            dsk[e >> 1] = Elem<T>::pack(d0, d1);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) pk[e] = dsk[e] = 0u;
        }
        // dS of chunk c lands in columns 16c .. 16c+15, whose scores have been read already
        tmem_st16(trow + S::COL_S + 16 * c, dsk);
        if (p.cls && j == 0) {                           // row of [P_0 | dS_0] for key block 0's gradients
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            *reinterpret_cast<uint4*>(sG + swz_off<128>(row, ch)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            *reinterpret_cast<uint4*>(sG + swz_off<128>(row, 4 + ch)) =
                make_uint4(dsk[4 * ch], dsk[4 * ch + 1], dsk[4 * ch + 2], dsk[4 * ch + 3]);
          }
          fence_proxy_async();                           // read by the tensor core (async proxy)
        }
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(ds_ready);
    }
    mbar_wait(dq_done, 0);
    tc_fence_after();
    T* dq = reinterpret_cast<T*>(p.dq) + b * p.dq_stride[0] + h * p.dq_stride[1] + (int64_t)qpos * p.dq_stride[2];
    d_store_row<T>(trow + S::COL_DQ, dq, qpos < p.L);
    if (p.cls) {
      // this tile's share of key block 0's gradients: TMEM lane = head column d, columns = keys
      const int d = row;
      float* part = p.gpart + (((int64_t)b * p.H + h) * p.T + t) * 2 * (kBlock * kDH);
#pragma unroll 1
      for (int which = 0; which < 2; ++which) {          // 0: dK_0 (Q^T dS_0, columns 32..63), 1: dV_0 (dO^T P_0, columns 0..31)
        uint32_t v[32];
        tmem_ld32(trow + (which == 0 ? S::COL_GK + 32 : S::COL_GV), v);
        tmem_wait_ld(v);
        float* dst = part + which * (kBlock * kDH) + d;
#pragma unroll
        for (int key = 0; key < kBlock; ++key) dst[key * kDH] = __uint_as_float(v[key]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------ dK/dV pass
template <typename T>
__global__ void __launch_bounds__(kDThreads, 1)
attn_d128_bwd_dkv_sm100_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                               const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO, const DParams p) {
  using S = DKvSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* kv_full = bars + 0;                // K and V
  uint64_t* q_full = bars + 1;                 // [2] Q and dO tile
  uint64_t* q_free = bars + 3;                 // [2]
  uint64_t* s_ready = bars + 5;                // S^T and dP^T of a query tile are in TMEM
  uint64_t* pds_ready = bars + 6;              // P^T and dS^T are in TMEM (128 arrivals)
  uint64_t* acc_done = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  float* sStat = reinterpret_cast<float*>(smem + S::OFF_STAT);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  // query blocks 4kt .. 4kt + left + 2 attend the tile's key blocks: query tiles kt .. kt + nc - 1
  int nc = (p.left + 3 + 3) / 4;
  if (kt + nc > p.T) nc = p.T - kt;

  if (threadIdx.x == 0) {
    mbar_init(kv_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(q_full + s, 1); mbar_init(q_free + s, 1); }
    mbar_init(s_ready, 1); mbar_init(pds_ready, 128); mbar_init(acc_done, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    if (lane == 0) { prefetch_tensormap(&tmK); prefetch_tensormap(&tmV); prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ---- TMA producer
    mbar_arrive_expect_tx_w(kv_full, 2 * kDTileB);
    d_load_tile(smem + S::OFF_K, &tmK, kv_full, kt * kTile, h, b);
    d_load_tile(smem + S::OFF_V, &tmV, kv_full, kt * kTile, h, b);
    for (int g = 0; g < nc; ++g) {
      const int s = g & 1;
      if (g >= 2) mbar_wait(q_free + s, ((g >> 1) - 1) & 1);
      mbar_arrive_expect_tx_w(q_full + s, 2 * kDTileB);
      d_load_tile(smem + S::OFF_Q + s * kDTileB, &tmQ, q_full + s, (kt + g) * kTile, h, b);
      d_load_tile(smem + S::OFF_DO + s * kDTileB, &tmDO, q_full + s, (kt + g) * kTile, h, b);
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S^T, dP^T of query tile g ; wait P^T, dS^T ; dV += P^T dO, dK += dS^T Q ; S^T, dP^T of tile g + 1
    const uint32_t idesc_s = make_idesc(kTile, kTile, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_o = make_idesc(kTile, kDH, Elem<T>::fmt, 0, 1);
    const uint32_t k_addr = smem_u32(smem + S::OFF_K), v_addr = smem_u32(smem + S::OFF_V);
    auto issue_sdp = [&](int g) {
      const int s = g & 1;
      mbar_wait(q_full + s, (g >> 1) & 1);
      tc_fence_after();
      const uint32_t q_addr = smem_u32(smem + S::OFF_Q + s * kDTileB), do_addr = smem_u32(smem + S::OFF_DO + s * kDTileB);
#pragma unroll
      for (int ks = 0; ks < kDH / 16; ++ks) {
        mma_ss_w(tmem_base + S::COL_S, kmajor_desc(k_addr, ks, kDHalf), kmajor_desc(q_addr, ks, kDHalf), idesc_s, ks > 0 ? 1u : 0u);
        mma_ss_w(tmem_base + S::COL_DP, kmajor_desc(v_addr, ks, kDHalf), kmajor_desc(do_addr, ks, kDHalf), idesc_s, ks > 0 ? 1u : 0u);
      }
      tc_commit_w(s_ready);
    };
    mbar_wait(kv_full, 0);
    issue_sdp(0);
    for (int g = 0; g < nc; ++g) {
      const int s = g & 1;
      mbar_wait(pds_ready, g & 1);
      tc_fence_after();
      const uint32_t q_addr = smem_u32(smem + S::OFF_Q + s * kDTileB), do_addr = smem_u32(smem + S::OFF_DO + s * kDTileB);
#pragma unroll
      for (int k2 = 0; k2 < kTile / 16; ++k2) {          // 16 queries per MMA; B = the dO / Q tile, MN-major
        mma_ts_w(tmem_base + S::COL_DV, tmem_base + S::COL_S + 8 * k2, mnmajor_desc(do_addr, k2, kDHalf), idesc_o, (g > 0 || k2 > 0) ? 1u : 0u);
        mma_ts_w(tmem_base + S::COL_DK, tmem_base + S::COL_DP + 8 * k2, mnmajor_desc(q_addr, k2, kDHalf), idesc_o, (g > 0 || k2 > 0) ? 1u : 0u);
      }
      tc_commit_w(q_free + s);
      if (g + 1 < nc) issue_sdp(g + 1);
      else tc_commit_w(acc_done);
    }
  } else {
    // ---- math warps: lane = key of block kb = 4kt + w, 128 query columns per tile
    const int row = warp * 32 + lane;
    const int kb = 4 * kt + warp;
    const int kpos = kt * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float kv = d_key_term(p, b, kpos);
    for (int g = 0; g < nc; ++g) {
      float* st = sStat + (g & 1) * 2 * kTile;
      {
        const int q = (kt + g) * kTile + (int)threadIdx.x;
        float nl = -INFINITY, nd = 0.f;                  // queries >= L: exact zeros in P^T and dS^T
        if (q < p.L) {
          const int64_t idx = ((int64_t)b * p.H + h) * p.L + q;
          nl = -p.lse[idx] * kLog2e;
          nd = -p.delta[idx] * p.scale;
        }
        st[threadIdx.x] = nl;
        st[kTile + threadIdx.x] = nd;
      }
      named_bar_sync(1, 128);
      mbar_wait(s_ready, g & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int qb = 4 * (kt + g) + c;
        const bool live = kb < p.nb && qb < p.nb && qb >= kb && qb <= kb + p.left - 1 && !(p.cls && kb == 0);
        uint32_t pk[16], dsk[16];
        if (live) {
          const bool diag = qb == kb;
          uint32_t sv[32], dv[32];
          tmem_ld32(trow + S::COL_S + 32 * c, sv);
          tmem_ld32(trow + S::COL_DP + 32 * c, dv);
          tmem_wait_ld(sv, dv);
          const float* nl = st + 32 * c;
          const float* nd = st + kTile + 32 * c;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float pe[2], de[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              pe[u] = fast_exp2(fmaf(__uint_as_float(sv[e + u]), p.scale_log2, nl[e + u]) + kv);
              if (diag && e + u < lane) pe[u] = 0.f;      // query before the key
              de[u] = pe[u] * fmaf(__uint_as_float(dv[e + u]), p.scale, nd[e + u]);
            }
            pk[e >> 1] = Elem<T>::pack(pe[0], pe[1]);
            dsk[e >> 1] = Elem<T>::pack(de[0], de[1]);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) pk[e] = dsk[e] = 0u;
        }
        tmem_st16(trow + S::COL_S + 16 * c, pk);
        tmem_st16(trow + S::COL_DP + 16 * c, dsk);
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(pds_ready);
    }
    mbar_wait(acc_done, 0);
    tc_fence_after();
    // key block 0 with the global column: written by the finish kernel from the dQ pass's partials
    const bool ok = kpos < p.L && !(p.cls && kb == 0);
    T* dv = reinterpret_cast<T*>(p.dv) + b * p.dv_stride[0] + h * p.dv_stride[1] + (int64_t)kpos * p.dv_stride[2];
    T* dk = reinterpret_cast<T*>(p.dk) + b * p.dk_stride[0] + h * p.dk_stride[1] + (int64_t)kpos * p.dk_stride[2];
    d_store_row<T>(trow + S::COL_DV, dv, ok);
    d_store_row<T>(trow + S::COL_DK, dk, ok);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem_base);
}

// dK / dV rows of key block 0 (include_cls): the sequence's per-query-tile partials summed in tile order
template <typename T>
__global__ void __launch_bounds__(256) attn_d128_bwd_finish_kernel(const DParams p) {
  // grid (2 * 32 * 128 / 256, B*H): one output element per thread
  const int seq = blockIdx.y, b = seq / p.H, h = seq % p.H;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int which = i / (kBlock * kDH), e = i % (kBlock * kDH), key = e / kDH, d = e % kDH;
  const float* src = p.gpart + (int64_t)seq * p.T * 2 * (kBlock * kDH) + which * (kBlock * kDH) + e;
  float part[8];
  float acc = 0.f;
  for (int t0 = 0; t0 < p.T; t0 += 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) part[k] = (t0 + k < p.T) ? __ldcg(src + (int64_t)(t0 + k) * 2 * (kBlock * kDH)) : 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc += part[k];          // fixed order: tile 0, 1, 2, ...
  }
  if (which == 0) reinterpret_cast<T*>(p.dk)[b * p.dk_stride[0] + h * p.dk_stride[1] + key * p.dk_stride[2] + d] = from_f32<T>(acc);
  else reinterpret_cast<T*>(p.dv)[b * p.dv_stride[0] + h * p.dv_stride[1] + key * p.dv_stride[2] + d] = from_f32<T>(acc);
}

// ------------------------------------------------------------------------------------------ host side
static size_t d_align256(size_t x) { return (x + 255) & ~size_t(255); }

bool d128_supported(const svae_attn_desc* d) {
  if (d->dtype != SVAE_DTYPE_BF16 && d->dtype != SVAE_DTYPE_F16) return false;
  if (d->head_dim != kDH || !(d->scale > 0.f) || !d->causal) return false;
  if (d->window_size < 1 || d->window_size > kDMaxLeft) return false;
  const int64_t tiles = ((int64_t)d->seq_len + kTile - 1) / kTile;
  return tiles <= INT32_MAX && d->heads <= 65535 && d->batch <= 65535;
}

size_t d128_bwd_workspace(const svae_attn_desc* d) {
  const size_t BH = (size_t)d->batch * d->heads, T = ((size_t)d->seq_len + kTile - 1) / kTile;
  const size_t delta = d_align256(sizeof(float) * BH * d->seq_len);
  return delta + (d->include_cls ? sizeof(float) * BH * T * 2 * kBlock * kDH : 0);
}

static DParams d_params(const svae_attn_desc* d, const float* kpm, float* lse) {
  const Band band = make_band(d->window_size, d->causal, d->include_cls);
  DParams p = {};
  p.kpm = kpm; p.lse = lse;
  p.L = d->seq_len; p.H = d->heads; p.T = (d->seq_len + kTile - 1) / kTile; p.nb = d->seq_len / kBlock;
  p.left = band.left; p.cls = band.cls;
  p.ns = band.cls + band.left + 3;
  p.ng = (p.ns + 3) / 4;
  p.scale = d->scale; p.scale_log2 = d->scale * kLog2e;
  return p;
}

template <typename T>
static int launch_d128_fwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out,
                           float* lse, cudaStream_t st) {
  CUtensorMap tmQ, tmK, tmV, tmO;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  const int L = d->seq_len, H = d->heads, B = d->batch;
  if ((rc = encode_tmap(&tmQ, dt, q, kDH, L, H, B, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, kDH, L, H, B, d->k_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, kDH, L, H, B, d->v_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmO, dt, out, kDH, L, H, B, d->o_stride, kTile))) return rc;
  const DParams p = d_params(d, kpm, lse);
  auto kern = attn_d128_fwd_sm100_kernel<T>;
  SVAE_CONFIGURE_SMEM(kern, DFwdSmem::DYN_BYTES);
  ScopedKernelTimer timer("attn_d128_fwd_sm100", st);
  kern<<<dim3(p.T, H, B), kDThreads, DFwdSmem::DYN_BYTES, st>>>(tmQ, tmK, tmV, tmO, p);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

template <typename T>
static int launch_d128_bwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out,
                           const void* dout, const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace,
                           cudaStream_t st) {
  CUtensorMap tmQ, tmDO, tmK32, tmV32, tmK, tmV;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  const int L = d->seq_len, H = d->heads, B = d->batch;
  if ((rc = encode_tmap(&tmQ, dt, q, kDH, L, H, B, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmDO, dt, dout, kDH, L, H, B, d->do_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK32, dt, k, kDH, L, H, B, d->k_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmV32, dt, v, kDH, L, H, B, d->v_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, kDH, L, H, B, d->k_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, kDH, L, H, B, d->v_stride, kTile))) return rc;
  DParams p = d_params(d, kpm, const_cast<float*>(lse));
  p.delta = reinterpret_cast<float*>(workspace);
  p.gpart = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + d_align256(sizeof(float) * (size_t)B * H * L));
  p.out = out; p.dout = dout; p.dq = dq; p.dk = dk; p.dv = dv;
  for (int i = 0; i < 3; ++i) {
    p.o_stride[i] = d->o_stride[i]; p.do_stride[i] = d->do_stride[i]; p.dq_stride[i] = d->dq_stride[i];
    p.dk_stride[i] = d->dk_stride[i]; p.dv_stride[i] = d->dv_stride[i];
  }
  auto kq = attn_d128_bwd_dq_sm100_kernel<T>;
  auto kkv = attn_d128_bwd_dkv_sm100_kernel<T>;
  SVAE_CONFIGURE_SMEM(kq, DDqSmem::DYN_BYTES);
  SVAE_CONFIGURE_SMEM(kkv, DKvSmem::DYN_BYTES);
  const dim3 grid(p.T, H, B);
  {
    ScopedKernelTimer timer("attn_d128_bwd_dq_sm100", st);
    kq<<<grid, kDThreads, DDqSmem::DYN_BYTES, st>>>(tmQ, tmDO, tmK32, tmV32, p);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  {
    ScopedKernelTimer timer("attn_d128_bwd_dkv_sm100", st);
    kkv<<<grid, kDThreads, DKvSmem::DYN_BYTES, st>>>(tmK, tmV, tmQ, tmDO, p);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  if (p.cls) {
    ScopedKernelTimer timer("attn_d128_bwd_finish", st);
    attn_d128_bwd_finish_kernel<T><<<dim3(2 * kBlock * kDH / 256, B * H), 256, 0, st>>>(p);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  return SVAE_OK;
}

#define SVAE_D128_SCOPE(fn)                                                                                                 \
  SVAE_REQUIRE(d128_supported(d), SVAE_ERR_UNSUPPORTED,                                                                    \
               fn ": head_dim 128 needs 16-bit tensors, a causal layout and window 1..%d (got dtype %d, causal %d, "      \
                  "window %d); non-causal head-128 layouts are not implemented",                                           \
               kDMaxLeft, d->dtype, d->causal, d->window_size)

int d128_fwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out, float* lse,
             cudaStream_t st) {
  SVAE_D128_SCOPE("sm100 attention forward");
  return d->dtype == SVAE_DTYPE_BF16 ? launch_d128_fwd<__nv_bfloat16>(d, q, k, v, kpm, out, lse, st)
                                     : launch_d128_fwd<__half>(d, q, k, v, kpm, out, lse, st);
}

int d128_bwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out, const void* dout,
             const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace, cudaStream_t st) {
  SVAE_D128_SCOPE("sm100 attention backward");
  return d->dtype == SVAE_DTYPE_BF16
             ? launch_d128_bwd<__nv_bfloat16>(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st)
             : launch_d128_bwd<__half>(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
}

#undef SVAE_D128_SCOPE

}  // namespace sm100
}  // namespace svae
