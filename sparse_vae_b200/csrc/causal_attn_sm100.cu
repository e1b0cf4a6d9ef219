// Dense CAUSAL self-attention with an additive key-padding mask for sm_100a (tcgen05 / TMEM / TMA): the self-attention
// of the non-sparse decoders (dense-benchmark, nonvae-wikipedia) in training, where every batch carries a padding mask.
//   out[b,h,i] = softmax_{j <= i}(scale * q_i . k_j + kpm[b, j]) v_j ,  lse[b,h,i] natural log, fp32.
// Keys j > i never enter the sum (masked by index, not by a large negative number), so a row whose keys 0..i are all
// padded spreads over keys 0..i and stays finite.
//
// Forward (one CTA per (128-query tile, head, batch), the last -- heaviest -- query tiles first; 6 warps): the forward
// of xattn_sm100.cu over the key tiles 0..t of query tile t.  Q stays in shared memory, K / V stream through a TMA ring,
// S = Q K^T double-buffered in TMEM, online softmax by four warps (one TMEM lane quarter each) with lazy rescaling of O,
// P written over S as 16-bit, O += P V accumulated in TMEM, O / l -> TMA store, LSE.  The causal mask costs a compare
// only on the diagonal tile; keys >= L are masked by index (the TMA unit zero-fills their rows).
//
// Backward: two passes, no atomics, bit-deterministic.  Both step through chunks of C rows (C = CPlan::kChunk).
//   dQ pass     one CTA per query tile t (heaviest first): Q, dO resident; the K / V chunks up to the tile's last key
//               streamed.  Per chunk S = Q K^T and dP = dO V^T (128 x C) into TMEM, dS = P o (dP - delta) * scale
//               written over S as 16-bit, dQ += dS K (A from TMEM).  delta = rowsum(dO o O) is computed here and
//               written for the second pass.
//   dK/dV pass  one CTA per key tile t (tile 0, the heaviest, first): K, V resident; the Q / dO chunks from the tile's
//               first key on streamed.  Per chunk S^T = K Q^T and dP^T = V dO^T (128 keys x C queries), P^T and dS^T
//               over them as 16-bit, dV += P^T dO, dK += dS^T Q.
//
// Head size 64 or 128, one implementation parameterised by DH (CPlan below).  A 128-column row is two SWIZZLE_128B
// atoms: operand tiles arrive as two TMA boxes of 64 columns, stored as two halves (attn_sm100.cuh, kmajor_desc /
// mnmajor_desc).  Per CTA (dynamic shared memory incl. barriers and alignment slack; TMEM columns allocated):
//                 head 64                                      head 128
//   forward       3 stages: 114 KB, 512 (S 2 x 128, O 64)       2 stages: 162 KB, 512 (S 2 x 128, O 128)
//   dQ pass       C = 64, 3 stages: 82 KB, 256 (S, dP 64, dQ 64)     C = 128, 2 stages: 195 KB, 512 (S, dP, dQ 128)
//   dK/dV pass    82 KB, 256 (S^T, dP^T, dV, dK 64)              195 KB, 512 (S^T, dP^T, dV, dK 128)
// At head 64 two backward CTAs share an SM and overlap each other's MMA / CUDA-core phases; at head 128 one CTA's
// shared memory rules that out, and 128-row chunks halve the hand-offs per byte instead (DESIGN 4.13b: measured against
// 64-row chunks and a 3-stage forward ring).
#include <type_traits>

#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kCThreads = 192;          // warps 0-3: softmax / math (one TMEM lane quarter each), 4: TMA, 5: MMA issue
constexpr float kCRescale = 8.0f;       // log2 units the running maximum may lag behind before O is rescaled

// per head size: forward K / V ring stages, backward rows per step (keys in the dQ pass, queries in the dK/dV pass),
// backward ring stages and backward CTAs per SM
template <int DH> struct CPlan;
template <> struct CPlan<64> { static constexpr int kFwdStages = 3, kChunk = 64, kBwdStages = 3, kBwdCtas = 2; };
template <> struct CPlan<128> { static constexpr int kFwdStages = 2, kChunk = 128, kBwdStages = 2, kBwdCtas = 1; };

constexpr int tmem_cols(int used) { return used <= 256 ? 256 : 512; }

template <int DH>
struct CFwdSmem {
  static constexpr int STAGES = CPlan<DH>::kFwdStages;
  static constexpr int HALF = kTile * 128;                        // one 64-column half of a tile: 16 KB
  static constexpr int TILE = kTile * DH * 2;                     // 16 / 32 KB
  static constexpr int OFF_Q = 0;                                 // later the output staging tile
  static constexpr int OFF_K = OFF_Q + TILE;                      // [STAGES]
  static constexpr int OFF_V = OFF_K + STAGES * TILE;             // [STAGES]
  static constexpr int OFF_KPM = OFF_V + STAGES * TILE;           // [2][128] additive key terms (log2 domain)
  static constexpr int OFF_BAR = OFF_KPM + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static_assert(DYN_BYTES <= 227 * 1024, "shared memory");
};

// both backward passes: a resident 128-row pair (Q, dO or K, V) and a ring of CH-row chunk pairs
template <int DH>
struct CBwdSmem {
  static constexpr int CH = CPlan<DH>::kChunk, STAGES = CPlan<DH>::kBwdStages;
  static constexpr int HALF_T = kTile * 128;                      // one 64-column half of a resident tile: 16 KB
  static constexpr int HALF_C = CH * 128;                         // one 64-column half of a chunk
  static constexpr int TILE = kTile * DH * 2;
  static constexpr int CHUNK = CH * DH * 2;
  static constexpr int OFF_A = 0;                                 // Q (dQ pass) / K (dK/dV pass)
  static constexpr int OFF_B = OFF_A + TILE;                      // dO / V
  static constexpr int OFF_C = OFF_B + TILE;                      // [STAGES] K / Q chunks
  static constexpr int OFF_D = OFF_C + STAGES * CHUNK;            // [STAGES] V / dO chunks
  static constexpr int OFF_STAT = OFF_D + STAGES * CHUNK;         // [2][2][CH] per-chunk terms (log2 domain)
  static constexpr int OFF_BAR = OFF_STAT + 4 * CH * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int COL_S = 0, COL_DP = CH, COL_ACC = 2 * CH;  // (dK/dV pass: dV at COL_ACC, dK at COL_ACC + DH)
  static constexpr int TMEM_DQ = tmem_cols(COL_ACC + DH), TMEM_DKV = tmem_cols(COL_ACC + 2 * DH);
  static_assert(CPlan<DH>::kBwdCtas * (DYN_BYTES + 1024) <= 228 * 1024, "backward CTAs per SM");
};

struct CParams {
  const float* kpm;     // [B, L] additive or null
  float* lse;           // [B, H, L] natural log
  float* delta;         // [B, H, L] rowsum(dO o O): written by the dQ pass, read by the dK/dV pass
  const void *out, *dout;
  void *dq, *dk, *dv;
  int64_t o_stride[3], do_stride[3], dq_stride[3], dk_stride[3], dv_stride[3];
  int L, H, BH, T;      // T = number of 128-row tiles
  float scale, scale_log2;
};

__device__ __forceinline__ float key_term(const CParams& p, int b, int key) {
  if (key >= p.L) return -INFINITY;
  return p.kpm ? p.kpm[(int64_t)b * p.L + key] * kLog2e : 0.f;
}

// DH fp32 TMEM columns of one row -> 16-bit -> global row (16-byte stores)
template <int DH, typename T>
__device__ __forceinline__ void store_row(uint32_t taddr, T* dst, bool ok) {
#pragma unroll
  for (int half = 0; half < DH / 32; ++half) {
    uint32_t v[32];
    tmem_ld32(taddr + 32 * half, v);
    tmem_wait_ld(v);
    if (ok) {
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        uint4 o;
        o.x = Elem<T>::pack(__uint_as_float(v[cq * 8 + 0]), __uint_as_float(v[cq * 8 + 1]));
        o.y = Elem<T>::pack(__uint_as_float(v[cq * 8 + 2]), __uint_as_float(v[cq * 8 + 3]));
        o.z = Elem<T>::pack(__uint_as_float(v[cq * 8 + 4]), __uint_as_float(v[cq * 8 + 5]));
        o.w = Elem<T>::pack(__uint_as_float(v[cq * 8 + 6]), __uint_as_float(v[cq * 8 + 7]));
        reinterpret_cast<uint4*>(dst)[half * 4 + cq] = o;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ forward
template <typename T, int DH>
__global__ void __launch_bounds__(kCThreads, 1)
causal_attn_fwd_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                             const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const CParams p) {
  using S = CFwdSmem<DH>;
  constexpr int kCStages = S::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;                 // [kCStages]
  uint64_t* v_full = bars + 1 + kCStages;      // [kCStages]
  uint64_t* kv_free = bars + 1 + 2 * kCStages; // [kCStages] both MMAs that read the stage have retired
  uint64_t* s_ready = bars + 1 + 3 * kCStages; // [2]
  uint64_t* p_ready = s_ready + 2;             // [2] (128 arrivals)
  uint64_t* o_done = p_ready + 2;              // P V of a tile retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 1);
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = p.T - 1 - (int)blockIdx.x / p.BH;      // heaviest query tiles first
  const int bh = (int)blockIdx.x % p.BH, h = bh % p.H, b = bh / p.H;
  const int nt = t + 1;                                // key tiles 0..t

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kCStages; ++s) { mbar_init(k_full + s, 1); mbar_init(v_full + s, 1); mbar_init(kv_free + s, 1); }
    for (int k = 0; k < 2; ++k) { mbar_init(s_ready + k, 1); mbar_init(p_ready + k, 128); }
    mbar_init(o_done, 1);
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
    // ---- TMA producer
    mbar_arrive_expect_tx_w(q_full, S::TILE);
    load_rows<DH>(smem + S::OFF_Q, S::HALF, &tmQ, q_full, t * kTile, h, b);    // rows >= L: zero-filled
    for (int i = 0; i < nt; ++i) {
      const int s = i % kCStages;
      if (i >= kCStages) mbar_wait(kv_free + s, ((i / kCStages) - 1) & 1);
      mbar_arrive_expect_tx_w(k_full + s, S::TILE);
      load_rows<DH>(smem + S::OFF_K + s * S::TILE, S::HALF, &tmK, k_full + s, i * kTile, h, b);
      mbar_arrive_expect_tx_w(v_full + s, S::TILE);
      load_rows<DH>(smem + S::OFF_V + s * S::TILE, S::HALF, &tmV, v_full + s, i * kTile, h, b);
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S(0); then per tile  S(i+1) ; wait P(i) ; O += P(i) V(i)   (in-order pipe: S(i+1) overwrites the
    //      buffer P(i-1) V(i-1) read only after that MMA)
    const uint32_t idesc_s = make_idesc(kTile, kTile, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_pv = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
    const uint32_t q_addr = smem_u32(smem + S::OFF_Q);
    auto issue_s = [&](int i) {
      const int s = i % kCStages;
      mbar_wait(k_full + s, (i / kCStages) & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * S::TILE);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks)
        mma_ss_w(tmem_base + 128 * (i & 1), kmajor_desc(q_addr, ks, S::HALF), kmajor_desc(k_addr, ks, S::HALF), idesc_s,
                 ks > 0 ? 1u : 0u);
      tc_commit_w(s_ready + (i & 1));
    };
    mbar_wait(q_full, 0);
    issue_s(0);
    for (int i = 0; i < nt; ++i) {
      if (i + 1 < nt) issue_s(i + 1);
      const int s = i % kCStages;
      mbar_wait(p_ready + (i & 1), (i >> 1) & 1);
      mbar_wait(v_full + s, (i / kCStages) & 1);
      tc_fence_after();
      const uint32_t v_addr = smem_u32(smem + S::OFF_V + s * S::TILE);
#pragma unroll
      for (int k2 = 0; k2 < kTile / 16; ++k2)          // 16 keys per MMA: A = P (16-bit, 8 columns), B = V rows MN-major
        mma_ts_w(tmem_base + COL_O, tmem_base + 128 * (i & 1) + 8 * k2, mnmajor_desc(v_addr, k2, S::HALF), idesc_pv,
                 (i > 0 || k2 > 0) ? 1u : 0u);
      tc_commit_w(o_done);
      tc_commit_w(kv_free + s);
    }
  } else {
    // ---- softmax / epilogue warps: warp w owns query rows 32 w .. 32 w + 31 of the tile
    const int row = warp * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    float m = -INFINITY, l = 0.f;                        // running maximum (log2 domain) and row sum relative to it
    for (int i = 0; i < nt; ++i) {
      float* kp = sKpm + (i & 1) * kTile;
      kp[threadIdx.x] = key_term(p, b, i * kTile + (int)threadIdx.x);
      named_bar_sync(1, 128);
      mbar_wait(s_ready + (i & 1), (i >> 1) & 1);
      tc_fence_after();
      const uint32_t ts = trow + 128 * (i & 1);
      // the diagonal tile (i == t) masks key columns > row; every other tile has no causal mask
      auto tile = [&](auto diag_c) {
        constexpr bool DIAG = decltype(diag_c)::value;
        // pass 1: maximum of the tile's scores
        float tmax = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t v[32];
          tmem_ld32(ts + 32 * c, v);
          tmem_wait_ld(v);
          const float4* k4 = reinterpret_cast<const float4*>(kp + 32 * c);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float4 kk = k4[e];
            const float kx[4] = {kk.x, kk.y, kk.z, kk.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float x = fmaf(__uint_as_float(v[4 * e + j]), p.scale_log2, kx[j]);
              if (DIAG && 32 * c + 4 * e + j > row) x = -INFINITY;
              tmax = fmaxf(tmax, x);
            }
          }
        }
        float alpha = 1.f;
        if (tmax > m + kCRescale || m == -INFINITY) {    // (also the first tile)
          alpha = (m == -INFINITY) ? 0.f : fast_exp2(m - tmax);
          m = tmax;
          l *= alpha;
        }
        const float neg_m = (m == -INFINITY) ? 0.f : -m;
        // pass 2: P = exp2(s * scale*log2e + mask - m) written over S as 16-bit, left to right
        float l0 = 0.f, l1 = 0.f;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t v[32], pk[16];
          tmem_ld32(ts + 32 * c, v);
          tmem_wait_ld(v);
          const float4* k4 = reinterpret_cast<const float4*>(kp + 32 * c);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float4 kk = k4[e];
            const float kx[4] = {kk.x, kk.y, kk.z, kk.w};
            float pe[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              pe[j] = fast_exp2(fmaf(__uint_as_float(v[4 * e + j]), p.scale_log2, kx[j]) + neg_m);
              if (DIAG && 32 * c + 4 * e + j > row) pe[j] = 0.f;
            }
            l0 += pe[0] + pe[2];
            l1 += pe[1] + pe[3];
            pk[2 * e] = Elem<T>::pack(pe[0], pe[1]);
            pk[2 * e + 1] = Elem<T>::pack(pe[2], pe[3]);
          }
          tmem_st16(ts + 16 * c, pk);
        }
        l += l0 + l1;
        return alpha;
      };
      const float alpha = (i == t) ? tile(std::true_type{}) : tile(std::false_type{});
      // lazy rescaling of the accumulator: O holds sums relative to the OLD maximum
      const bool any = __any_sync(0xffffffffu, alpha != 1.f);
      if (any && i > 0) {
        mbar_wait(o_done, (i - 1) & 1);                 // P V of the previous tile has retired
        tc_fence_after();
#pragma unroll 1
        for (int half = 0; half < DH / 32; ++half) {
          uint32_t o[32];
          tmem_ld32(trow + COL_O + 32 * half, o);
          tmem_wait_ld(o);
#pragma unroll
          for (int e = 0; e < 32; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
          uint32_t lo[16], hi[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) { lo[e] = o[e]; hi[e] = o[16 + e]; }
          tmem_st16(trow + COL_O + 32 * half, lo);
          tmem_st16(trow + COL_O + 32 * half + 16, hi);
        }
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_ready + (i & 1));
    }
    // epilogue: O / l -> 16-bit -> swizzled staging (the Q tile, DH / 64 halves) -> TMA store ; LSE
    mbar_wait(o_done, (nt - 1) & 1);
    tc_fence_after();
    uint8_t* stage = smem + S::OFF_Q;
    const float inv = 1.0f / l;
#pragma unroll
    for (int half = 0; half < DH / 32; ++half) {
      uint32_t o[32];
      tmem_ld32(trow + COL_O + 32 * half, o);
      tmem_wait_ld(o);
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        uint4 w4;
        w4.x = Elem<T>::pack(__uint_as_float(o[cq * 8 + 0]) * inv, __uint_as_float(o[cq * 8 + 1]) * inv);
        w4.y = Elem<T>::pack(__uint_as_float(o[cq * 8 + 2]) * inv, __uint_as_float(o[cq * 8 + 3]) * inv);
        w4.z = Elem<T>::pack(__uint_as_float(o[cq * 8 + 4]) * inv, __uint_as_float(o[cq * 8 + 5]) * inv);
        w4.w = Elem<T>::pack(__uint_as_float(o[cq * 8 + 6]) * inv, __uint_as_float(o[cq * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(stage + (half >> 1) * S::HALF + swz_off<128>(row, (half & 1) * 4 + cq)) = w4;
      }
    }
    const int qpos = t * kTile + row;
    if (qpos < p.L) p.lse[((int64_t)b * p.H + h) * p.L + qpos] = (m + log2f(l)) * kLn2;
    fence_proxy_async();
    named_bar_sync(1, 128);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int c = 0; c < DH / 64; ++c)                // rows >= L are outside the tensor: clipped
        tma_store_4d(&tmO, stage + c * S::HALF, 64 * c, t * kTile, h, b);
      tma_store_commit();
      tma_store_wait_all();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------ dQ pass
template <typename T, int DH>
__global__ void __launch_bounds__(kCThreads, CPlan<DH>::kBwdCtas)
causal_attn_bwd_dq_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                                const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV, const CParams p) {
  using S = CBwdSmem<DH>;
  constexpr int kChunk = S::CH, kCStages = S::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;                 // Q and dO
  uint64_t* kv_full = bars + 1;                // [kCStages] K and V chunk
  uint64_t* kv_free = bars + 1 + kCStages;     // [kCStages] the MMAs that read the stage have retired
  uint64_t* s_ready = bars + 1 + 2 * kCStages; // S and dP of a chunk are in TMEM
  uint64_t* ds_ready = s_ready + 1;            // dS of a chunk is in TMEM (128 arrivals)
  uint64_t* dq_done = ds_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dq_done + 1);
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_STAT);       // [2][kChunk]

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = p.T - 1 - (int)blockIdx.x / p.BH;      // heaviest query tiles first
  const int bh = (int)blockIdx.x % p.BH, h = bh % p.H, b = bh / p.H;
  const int nlim = (p.L + kChunk - 1) / kChunk;
  const int nupto = (t + 1) * (kTile / kChunk);                   // key chunks up to the diagonal tile's last key
  const int nc = nupto < nlim ? nupto : nlim;                     // ... that hold a key < L

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kCStages; ++s) { mbar_init(kv_full + s, 1); mbar_init(kv_free + s, 1); }
    mbar_init(s_ready, 1); mbar_init(ds_ready, 128); mbar_init(dq_done, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    if (lane == 0) { prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV); }
    tmem_alloc<S::TMEM_DQ>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ---- TMA producer
    mbar_arrive_expect_tx_w(q_full, 2 * S::TILE);
    load_rows<DH>(smem + S::OFF_A, S::HALF_T, &tmQ, q_full, t * kTile, h, b);
    load_rows<DH>(smem + S::OFF_B, S::HALF_T, &tmDO, q_full, t * kTile, h, b);
    for (int j = 0; j < nc; ++j) {
      const int s = j % kCStages;
      if (j >= kCStages) mbar_wait(kv_free + s, ((j / kCStages) - 1) & 1);
      mbar_arrive_expect_tx_w(kv_full + s, 2 * S::CHUNK);
      load_rows<DH>(smem + S::OFF_C + s * S::CHUNK, S::HALF_C, &tmK, kv_full + s, j * kChunk, h, b);
      load_rows<DH>(smem + S::OFF_D + s * S::CHUNK, S::HALF_C, &tmV, kv_full + s, j * kChunk, h, b);
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S, dP of chunk j ; wait dS(j) ; dQ += dS(j) K(j) ; S, dP of chunk j + 1 (in-order pipe: they
    //      overwrite dS(j) only after the dQ MMAs read it)
    const uint32_t idesc_s = make_idesc(kTile, kChunk, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_dq = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
    const uint32_t q_addr = smem_u32(smem + S::OFF_A), do_addr = smem_u32(smem + S::OFF_B);
    auto issue_sdp = [&](int j) {
      const int s = j % kCStages;
      mbar_wait(kv_full + s, (j / kCStages) & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_C + s * S::CHUNK), v_addr = smem_u32(smem + S::OFF_D + s * S::CHUNK);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        mma_ss_w(tmem_base + S::COL_S, kmajor_desc(q_addr, ks, S::HALF_T), kmajor_desc(k_addr, ks, S::HALF_C), idesc_s,
                 ks > 0 ? 1u : 0u);
        mma_ss_w(tmem_base + S::COL_DP, kmajor_desc(do_addr, ks, S::HALF_T), kmajor_desc(v_addr, ks, S::HALF_C), idesc_s,
                 ks > 0 ? 1u : 0u);
      }
      tc_commit_w(s_ready);
    };
    mbar_wait(q_full, 0);
    issue_sdp(0);
    for (int j = 0; j < nc; ++j) {
      const int s = j % kCStages;
      mbar_wait(ds_ready, j & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_C + s * S::CHUNK);
#pragma unroll
      for (int k2 = 0; k2 < kChunk / 16; ++k2)         // 16 keys per MMA: A = dS (16-bit, 8 columns), B = K rows MN-major
        mma_ts_w(tmem_base + S::COL_ACC, tmem_base + S::COL_S + 8 * k2, mnmajor_desc(k_addr, k2, S::HALF_C), idesc_dq,
                 (j > 0 || k2 > 0) ? 1u : 0u);
      tc_commit_w(kv_free + s);
      if (j + 1 < nc) issue_sdp(j + 1);
      else tc_commit_w(dq_done);
    }
  } else {
    // ---- math warps: warp w owns query rows 32 w .. 32 w + 31 of the tile
    const int row = warp * 32 + lane;
    const int qpos = t * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    const int64_t stat_idx = ((int64_t)b * p.H + h) * p.L + qpos;
    // delta = rowsum(dO o O) straight from global memory; rows >= L (zero Q and dO) get neutral statistics
    float nl = 0.f, nd = 0.f;
    if (qpos < p.L) {
      const T* o = reinterpret_cast<const T*>(p.out) + b * p.o_stride[0] + h * p.o_stride[1] + (int64_t)qpos * p.o_stride[2];
      const T* d_o = reinterpret_cast<const T*>(p.dout) + b * p.do_stride[0] + h * p.do_stride[1] + (int64_t)qpos * p.do_stride[2];
      float d = 0.f;
#pragma unroll
      for (int ch = 0; ch < DH / 8; ++ch) {
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
    for (int j = 0; j < nc; ++j) {
      float* kp = sKpm + (j & 1) * kChunk;
      if (threadIdx.x < kChunk) kp[threadIdx.x] = key_term(p, b, j * kChunk + (int)threadIdx.x);
      named_bar_sync(1, 128);
      mbar_wait(s_ready, j & 1);
      tc_fence_after();
      const int rel = j * kChunk - t * kTile;           // key column c is key rel + c of the tile's row numbering
      auto chunk = [&](auto diag_c) {
        constexpr bool DIAG = decltype(diag_c)::value;
#pragma unroll
        for (int half = 0; half < kChunk / 32; ++half) {
          uint32_t sv[32], dv[32], dsk[16];
          tmem_ld32(trow + S::COL_S + 32 * half, sv);
          tmem_ld32(trow + S::COL_DP + 32 * half, dv);
          tmem_wait_ld(sv, dv);
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float pe[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              pe[u] = fast_exp2(fmaf(__uint_as_float(sv[e + u]), p.scale_log2, kp[32 * half + e + u]) + nl);
              if (DIAG && rel + 32 * half + e + u > row) pe[u] = 0.f;
            }
            const float d0 = pe[0] * fmaf(__uint_as_float(dv[e]), p.scale, nd);
            const float d1 = pe[1] * fmaf(__uint_as_float(dv[e + 1]), p.scale, nd);
            dsk[e >> 1] = Elem<T>::pack(d0, d1);
          }
          // dS of half n lands in columns 16n .. 16n+15, whose scores have been read already
          tmem_st16(trow + S::COL_S + 16 * half, dsk);
        }
      };
      if (rel + kChunk - 1 > 0) chunk(std::true_type{});          // some key of the chunk lies past some row
      else chunk(std::false_type{});
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(ds_ready);
    }
    mbar_wait(dq_done, 0);
    tc_fence_after();
    T* dq = reinterpret_cast<T*>(p.dq) + b * p.dq_stride[0] + h * p.dq_stride[1] + (int64_t)qpos * p.dq_stride[2];
    store_row<DH, T>(trow + S::COL_ACC, dq, qpos < p.L);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<S::TMEM_DQ>(tmem_base);
}

// ------------------------------------------------------------------------------------------ dK/dV pass
template <typename T, int DH>
__global__ void __launch_bounds__(kCThreads, CPlan<DH>::kBwdCtas)
causal_attn_bwd_dkv_sm100_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                                 const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO, const CParams p) {
  using S = CBwdSmem<DH>;
  constexpr int kChunk = S::CH, kCStages = S::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* kv_full = bars + 0;                // K and V
  uint64_t* q_full = bars + 1;                 // [kCStages] Q and dO chunk
  uint64_t* q_free = bars + 1 + kCStages;      // [kCStages]
  uint64_t* s_ready = bars + 1 + 2 * kCStages; // S^T and dP^T of a chunk are in TMEM
  uint64_t* pds_ready = s_ready + 1;           // P^T and dS^T of a chunk are in TMEM (128 arrivals)
  uint64_t* acc_done = pds_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_done + 1);
  float* sStat = reinterpret_cast<float*>(smem + S::OFF_STAT);      // [2][-lse*log2e (kChunk) | -delta*scale (kChunk)]

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = (int)blockIdx.x / p.BH;                // key tile 0 (every query attends it) first
  const int bh = (int)blockIdx.x % p.BH, h = bh % p.H, b = bh / p.H;
  const int c0 = t * (kTile / kChunk);                 // first query chunk that can attend the tile
  const int nc = (p.L + kChunk - 1) / kChunk - c0;

  if (threadIdx.x == 0) {
    mbar_init(kv_full, 1);
    for (int s = 0; s < kCStages; ++s) { mbar_init(q_full + s, 1); mbar_init(q_free + s, 1); }
    mbar_init(s_ready, 1); mbar_init(pds_ready, 128); mbar_init(acc_done, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    if (lane == 0) { prefetch_tensormap(&tmK); prefetch_tensormap(&tmV); prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); }
    tmem_alloc<S::TMEM_DKV>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ---- TMA producer
    mbar_arrive_expect_tx_w(kv_full, 2 * S::TILE);
    load_rows<DH>(smem + S::OFF_A, S::HALF_T, &tmK, kv_full, t * kTile, h, b);
    load_rows<DH>(smem + S::OFF_B, S::HALF_T, &tmV, kv_full, t * kTile, h, b);
    for (int j = 0; j < nc; ++j) {
      const int s = j % kCStages;
      if (j >= kCStages) mbar_wait(q_free + s, ((j / kCStages) - 1) & 1);
      mbar_arrive_expect_tx_w(q_full + s, 2 * S::CHUNK);
      load_rows<DH>(smem + S::OFF_C + s * S::CHUNK, S::HALF_C, &tmQ, q_full + s, (c0 + j) * kChunk, h, b);
      load_rows<DH>(smem + S::OFF_D + s * S::CHUNK, S::HALF_C, &tmDO, q_full + s, (c0 + j) * kChunk, h, b);
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S^T, dP^T of chunk j ; wait P^T, dS^T ; dV += P^T dO, dK += dS^T Q ; S^T, dP^T of chunk j + 1
    const uint32_t idesc_s = make_idesc(kTile, kChunk, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_o = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
    const uint32_t k_addr = smem_u32(smem + S::OFF_A), v_addr = smem_u32(smem + S::OFF_B);
    auto issue_sdp = [&](int j) {
      const int s = j % kCStages;
      mbar_wait(q_full + s, (j / kCStages) & 1);
      tc_fence_after();
      const uint32_t q_addr = smem_u32(smem + S::OFF_C + s * S::CHUNK), do_addr = smem_u32(smem + S::OFF_D + s * S::CHUNK);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        mma_ss_w(tmem_base + S::COL_S, kmajor_desc(k_addr, ks, S::HALF_T), kmajor_desc(q_addr, ks, S::HALF_C), idesc_s,
                 ks > 0 ? 1u : 0u);
        mma_ss_w(tmem_base + S::COL_DP, kmajor_desc(v_addr, ks, S::HALF_T), kmajor_desc(do_addr, ks, S::HALF_C), idesc_s,
                 ks > 0 ? 1u : 0u);
      }
      tc_commit_w(s_ready);
    };
    mbar_wait(kv_full, 0);
    issue_sdp(0);
    for (int j = 0; j < nc; ++j) {
      const int s = j % kCStages;
      mbar_wait(pds_ready, j & 1);
      tc_fence_after();
      const uint32_t q_addr = smem_u32(smem + S::OFF_C + s * S::CHUNK), do_addr = smem_u32(smem + S::OFF_D + s * S::CHUNK);
#pragma unroll
      for (int ks = 0; ks < kChunk / 16; ++ks) {       // 16 queries per MMA; B = the dO / Q chunk rows, MN-major
        mma_ts_w(tmem_base + S::COL_ACC, tmem_base + S::COL_S + 8 * ks, mnmajor_desc(do_addr, ks, S::HALF_C), idesc_o,
                 (j > 0 || ks > 0) ? 1u : 0u);
        mma_ts_w(tmem_base + S::COL_ACC + DH, tmem_base + S::COL_DP + 8 * ks, mnmajor_desc(q_addr, ks, S::HALF_C), idesc_o,
                 (j > 0 || ks > 0) ? 1u : 0u);
      }
      tc_commit_w(q_free + s);
      if (j + 1 < nc) issue_sdp(j + 1);
      else tc_commit_w(acc_done);
    }
  } else {
    // ---- math warps: lane = key row of the tile, 64 query columns per chunk
    const int row = warp * 32 + lane;
    const int kpos = t * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float kv = key_term(p, b, kpos);
    for (int j = 0; j < nc; ++j) {
      float* st = sStat + (j & 1) * 2 * kChunk;
      if (threadIdx.x < kChunk) {
        const int q = (c0 + j) * kChunk + (int)threadIdx.x;
        float nl = -INFINITY, nd = 0.f;                  // queries >= L: exact zeros in P^T and dS^T
        if (q < p.L) {
          const int64_t idx = ((int64_t)b * p.H + h) * p.L + q;
          nl = -p.lse[idx] * kLog2e;
          nd = -p.delta[idx] * p.scale;
        }
        st[threadIdx.x] = nl;
        st[kChunk + threadIdx.x] = nd;
      }
      named_bar_sync(1, 128);
      mbar_wait(s_ready, j & 1);
      tc_fence_after();
      const int rel = j * kChunk;                        // query column c is query rel + c of the tile's key numbering
      auto chunk = [&](auto diag_c) {
        constexpr bool DIAG = decltype(diag_c)::value;
#pragma unroll
        for (int half = 0; half < kChunk / 32; ++half) {
          uint32_t sv[32], dv[32], pk[16], dsk[16];
          tmem_ld32(trow + S::COL_S + 32 * half, sv);
          tmem_ld32(trow + S::COL_DP + 32 * half, dv);
          tmem_wait_ld(sv, dv);
          const float* nl = st + 32 * half;
          const float* nd = st + kChunk + 32 * half;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float pe[2], de[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              pe[u] = fast_exp2(fmaf(__uint_as_float(sv[e + u]), p.scale_log2, nl[e + u]) + kv);
              if (DIAG && rel + 32 * half + e + u < row) pe[u] = 0.f;     // query before the key
              de[u] = pe[u] * fmaf(__uint_as_float(dv[e + u]), p.scale, nd[e + u]);
            }
            pk[e >> 1] = Elem<T>::pack(pe[0], pe[1]);
            dsk[e >> 1] = Elem<T>::pack(de[0], de[1]);
          }
          tmem_st16(trow + S::COL_S + 16 * half, pk);
          tmem_st16(trow + S::COL_DP + 16 * half, dsk);
        }
      };
      if (rel < kTile - 1) chunk(std::true_type{});      // the chunks of query tile t hold queries before some key
      else chunk(std::false_type{});
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(pds_ready);
    }
    mbar_wait(acc_done, 0);
    tc_fence_after();
    T* dv = reinterpret_cast<T*>(p.dv) + b * p.dv_stride[0] + h * p.dv_stride[1] + (int64_t)kpos * p.dv_stride[2];
    T* dk = reinterpret_cast<T*>(p.dk) + b * p.dk_stride[0] + h * p.dk_stride[1] + (int64_t)kpos * p.dk_stride[2];
    store_row<DH, T>(trow + S::COL_ACC, dv, kpos < p.L);
    store_row<DH, T>(trow + S::COL_ACC + DH, dk, kpos < p.L);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<S::TMEM_DKV>(tmem_base);
}

// ------------------------------------------------------------------------------------------ host side
static size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

bool causal_supported(const svae_xattn_desc* d) {
  if (d->dtype != SVAE_DTYPE_BF16 && d->dtype != SVAE_DTYPE_F16) return false;
  if ((d->head_dim != 64 && d->head_dim != 128) || !(d->scale > 0.f) || d->batch < 1 || d->heads < 1) return false;
  if (d->num_queries != d->num_keys || d->num_keys < 1) return false;
  const int64_t tiles = ((int64_t)d->num_keys + kTile - 1) / kTile;
  return tiles * d->batch * d->heads <= INT32_MAX;
}

size_t causal_workspace(const svae_xattn_desc* d) { return align256(sizeof(float) * (size_t)d->batch * d->heads * d->num_keys); }

static CParams causal_params(const svae_xattn_desc* d, const float* kpm, float* lse) {
  CParams p = {};
  p.kpm = kpm; p.lse = lse;
  p.L = d->num_keys; p.H = d->heads; p.BH = d->batch * d->heads; p.T = (d->num_keys + kTile - 1) / kTile;
  p.scale = d->scale; p.scale_log2 = d->scale * kLog2e;
  return p;
}

template <typename T, int DH>
static int launch_causal_fwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out,
                             float* lse, cudaStream_t st) {
  CUtensorMap tmQ, tmK, tmV, tmO;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  const int L = d->num_keys;
  if ((rc = encode_tmap(&tmQ, dt, q, DH, L, d->heads, d->batch, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, DH, L, d->heads, d->batch, d->k_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, DH, L, d->heads, d->batch, d->v_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmO, dt, out, DH, L, d->heads, d->batch, d->o_stride, kTile))) return rc;
  const CParams p = causal_params(d, kpm, lse);
  auto kern = causal_attn_fwd_sm100_kernel<T, DH>;
  SVAE_CONFIGURE_SMEM(kern, CFwdSmem<DH>::DYN_BYTES);
  ScopedKernelTimer timer("causal_attn_fwd_sm100", st);
  kern<<<p.T * p.BH, kCThreads, CFwdSmem<DH>::DYN_BYTES, st>>>(tmQ, tmK, tmV, tmO, p);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

template <typename T, int DH>
static int launch_causal_bwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v, const void* out,
                             const void* dout, const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace,
                             cudaStream_t st) {
  using S = CBwdSmem<DH>;
  constexpr int kChunk = S::CH;
  CUtensorMap tmQ, tmDO, tmKc, tmVc, tmK, tmV, tmQc, tmDOc;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  const int L = d->num_keys, H = d->heads, B = d->batch;
  if ((rc = encode_tmap(&tmQ, dt, q, DH, L, H, B, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmDO, dt, dout, DH, L, H, B, d->do_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmKc, dt, k, DH, L, H, B, d->k_stride, kChunk))) return rc;
  if ((rc = encode_tmap(&tmVc, dt, v, DH, L, H, B, d->v_stride, kChunk))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, DH, L, H, B, d->k_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, DH, L, H, B, d->v_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmQc, dt, q, DH, L, H, B, d->q_stride, kChunk))) return rc;
  if ((rc = encode_tmap(&tmDOc, dt, dout, DH, L, H, B, d->do_stride, kChunk))) return rc;
  CParams p = causal_params(d, kpm, const_cast<float*>(lse));
  p.delta = reinterpret_cast<float*>(workspace);
  p.out = out; p.dout = dout; p.dq = dq; p.dk = dk; p.dv = dv;
  for (int i = 0; i < 3; ++i) {
    p.o_stride[i] = d->o_stride[i]; p.do_stride[i] = d->do_stride[i]; p.dq_stride[i] = d->dq_stride[i];
    p.dk_stride[i] = d->dk_stride[i]; p.dv_stride[i] = d->dv_stride[i];
  }
  auto kq = causal_attn_bwd_dq_sm100_kernel<T, DH>;
  auto kkv = causal_attn_bwd_dkv_sm100_kernel<T, DH>;
  SVAE_CONFIGURE_SMEM(kq, S::DYN_BYTES);
  SVAE_CONFIGURE_SMEM(kkv, S::DYN_BYTES);
  {
    ScopedKernelTimer timer("causal_attn_bwd_dq_sm100", st);
    kq<<<p.T * p.BH, kCThreads, S::DYN_BYTES, st>>>(tmQ, tmDO, tmKc, tmVc, p);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  {
    ScopedKernelTimer timer("causal_attn_bwd_dkv_sm100", st);
    kkv<<<p.T * p.BH, kCThreads, S::DYN_BYTES, st>>>(tmK, tmV, tmQc, tmDOc, p);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

}  // namespace sm100
}  // namespace svae

using namespace svae;

static bool c_tma_ok(const void* p, const int64_t s[3]) {
  return reinterpret_cast<uintptr_t>(p) % 16 == 0 && (s[0] * 2) % 16 == 0 && (s[1] * 2) % 16 == 0 && (s[2] * 2) % 16 == 0;
}

#define SVAE_CAUSAL_SCOPE(fn)                                                                                               \
  SVAE_REQUIRE(sm100::causal_supported(d), SVAE_ERR_UNSUPPORTED,                                                           \
               fn ": needs 16-bit tensors, head_dim 64 or 128 and num_queries == num_keys >= 1 (got dtype %d, head_dim "   \
                  "%d, %d queries, %d keys)",                                                                               \
               d->dtype, d->head_dim, d->num_queries, d->num_keys)

extern "C" int svae_causal_attn_supported(const svae_xattn_desc* d) { return d && sm100::causal_supported(d) ? 1 : 0; }

extern "C" int svae_causal_attn_fwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v,
                                    const float* key_padding_mask, void* out, float* lse, void* stream) {
  SVAE_REQUIRE(d && q && k && v && out && lse, SVAE_ERR_INVALID, "svae_causal_attn_fwd: null argument");
  SVAE_CAUSAL_SCOPE("svae_causal_attn_fwd");
  SVAE_REQUIRE(c_tma_ok(q, d->q_stride) && c_tma_ok(k, d->k_stride) && c_tma_ok(v, d->v_stride) && c_tma_ok(out, d->o_stride),
               SVAE_ERR_UNSUPPORTED, "svae_causal_attn_fwd: tensors must be 16-byte aligned with strides that are multiples of 8 elements");
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool bf16 = d->dtype == SVAE_DTYPE_BF16;
  if (d->head_dim == 128)
    return bf16 ? sm100::launch_causal_fwd<__nv_bfloat16, 128>(d, q, k, v, key_padding_mask, out, lse, st)
                : sm100::launch_causal_fwd<__half, 128>(d, q, k, v, key_padding_mask, out, lse, st);
  return bf16 ? sm100::launch_causal_fwd<__nv_bfloat16, 64>(d, q, k, v, key_padding_mask, out, lse, st)
              : sm100::launch_causal_fwd<__half, 64>(d, q, k, v, key_padding_mask, out, lse, st);
}

extern "C" size_t svae_causal_attn_bwd_workspace_bytes(const svae_xattn_desc* d) {
  return d && sm100::causal_supported(d) ? sm100::causal_workspace(d) : 0;
}

extern "C" int svae_causal_attn_bwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v, const void* out,
                                    const void* dout, const float* lse, const float* key_padding_mask, void* dq, void* dk, void* dv,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  SVAE_REQUIRE(d && q && k && v && out && dout && lse && dq && dk && dv, SVAE_ERR_INVALID, "svae_causal_attn_bwd: null argument");
  SVAE_CAUSAL_SCOPE("svae_causal_attn_bwd");
  SVAE_REQUIRE(c_tma_ok(q, d->q_stride) && c_tma_ok(k, d->k_stride) && c_tma_ok(v, d->v_stride) && c_tma_ok(out, d->o_stride) &&
                   c_tma_ok(dout, d->do_stride) && c_tma_ok(dq, d->dq_stride) && c_tma_ok(dk, d->dk_stride) &&
                   c_tma_ok(dv, d->dv_stride),
               SVAE_ERR_UNSUPPORTED, "svae_causal_attn_bwd: tensors must be 16-byte aligned with strides that are multiples of 8 elements");
  SVAE_REQUIRE(workspace && workspace_bytes >= sm100::causal_workspace(d), SVAE_ERR_INVALID,
               "svae_causal_attn_bwd: workspace of %zu bytes, %zu needed", workspace_bytes, sm100::causal_workspace(d));
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool bf16 = d->dtype == SVAE_DTYPE_BF16;
  if (d->head_dim == 128)
    return bf16 ? sm100::launch_causal_bwd<__nv_bfloat16, 128>(d, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, workspace, st)
                : sm100::launch_causal_bwd<__half, 128>(d, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, workspace, st);
  return bf16 ? sm100::launch_causal_bwd<__nv_bfloat16, 64>(d, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, workspace, st)
              : sm100::launch_causal_bwd<__half, 64>(d, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, workspace, st);
}
