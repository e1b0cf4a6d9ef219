// Dense attention of a FEW queries over a LONG key sequence for sm_100a (tcgen05 / TMEM / TMA): the Perceiver encoder's
// learned-query layers (64 latents attending all L tokens of every sample; reference core/perceiver.py:16-50 through
// core/attention.py:83-100, non-causal, additive key padding -1e7).  cuDNN / flash kernels treat this as a generic
// attention problem with 64x128 tiles (142 us forward, 196 us backward per call at 16 x 4096 tokens on an sm_80 code
// path); here it is what it is: K and V streamed through shared memory ONCE (134 MB per call), everything else on chip.
//
// Forward (one CTA per (batch, head), 6 warps): Q (<= 128 rows, zero-filled above nq by the TMA box) stays in shared
// memory; per 128-key tile  S = Q K^T (tcgen05, fp32 in TMEM, two buffers) -> online softmax in the log2 domain by
// the warps that own valid query rows (two passes over TMEM per tile, lazy rescaling of O: only when the running
// maximum grows by more than 2^8) -> P written over S as 16-bit -> O += P V (A from TMEM) -> O / l -> TMA store, LSE.
// Backward (one CTA per (batch, head), 16 warps, the machinery of attn_bwd1_sm100.cu without sparsity): per key tile
// S^T = K Q^T and dP^T = V dO^T (128 keys x nq queries) -> P^T, dS^T as 16-bit TMEM operands -> dV = P^T dO and
// dK = dS^T Q stored per tile; dS^T also staged in shared memory for dQ += dS K, whose accumulator lives in TMEM for
// the whole sequence.  No atomics: bit-deterministic.
// Key splits (grid (B*H) x splits): below 64 (batch, head) pairs one CTA per pair leaves most SMs idle, so split s of a
// pair takes a contiguous, balanced run of the 128-key tiles; only its TMA coordinates, key-mask staging and
// "key >= Lk" test move.  With several splits the forward writes O_s / l_s, m_s and l_s in fp32 and
// xattn_fwd_merge_kernel combines them in split order; the backward (merged lse, delta recomputed per CTA) stores dK / dV
// of its own tiles and drains its partial dQ in fp32, which xattn_dq_reduce_kernel sums in split order.  One split
// launches exactly the one-CTA-per-pair kernels above.
// HBM roofline: forward reads K, V once; backward reads K, V and writes dK, dV once.
#include <algorithm>

#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kXThreads = 192;
constexpr int kXStages = 3;
constexpr float kXRescale = 8.0f;       // log2 units the running maximum may lag behind before O is rescaled

template <int DH>
struct XFwdSmem {
  static constexpr int ROWB = DH * 2;
  static constexpr int TILE = kTile * ROWB;                       // 16 KB
  static constexpr int OFF_Q = 0;                                 // later the output staging tile
  static constexpr int OFF_K = OFF_Q + TILE;                      // [kXStages]
  static constexpr int OFF_V = OFF_K + kXStages * TILE;           // [kXStages]
  static constexpr int OFF_KPM = OFF_V + kXStages * TILE;         // [2][128] additive key terms (log2 domain)
  static constexpr int OFF_BAR = OFF_KPM + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
};

struct XParams {
  const float* kpm;     // [B, Lk] additive or null
  float* lse;           // [B, H, nq] natural log
  const float* delta;   // backward: unused (computed in the kernel)
  float* part_o;        // key_splits > 1: [B*H][splits][nq][DH] the split's O_s / l_s, fp32
  float* part_m;        // key_splits > 1: [B*H][splits][nq] the split's running maximum m_s (log2 domain)
  float* part_l;        // key_splits > 1: [B*H][splits][nq] the split's row sum l_s relative to m_s
  int nq, Lk, H;
  float scale, scale_log2;
};

// key tiles [first, last) of split s of `splits` over nt tiles: contiguous, balanced to one tile, never empty (splits <= nt)
__device__ __forceinline__ void x_split_tiles(int nt, int splits, int s, int& first, int& last) {
  first = (int)((int64_t)s * nt / splits);
  last = (int)((int64_t)(s + 1) * nt / splits);
}

template <typename T, int DH>
__global__ void __launch_bounds__(kXThreads, 1)
xattn_fwd_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                       const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const XParams p) {
  using S = XFwdSmem<DH>;
  constexpr int ROWB = S::ROWB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;                 // [kXStages]
  uint64_t* v_full = bars + 1 + kXStages;      // [kXStages]
  uint64_t* kv_free = bars + 1 + 2 * kXStages; // [kXStages] both MMAs that read the stage have retired
  uint64_t* s_ready = bars + 1 + 3 * kXStages; // [2]
  uint64_t* p_ready = s_ready + 2;             // [2] (128 arrivals)
  uint64_t* o_done = p_ready + 2;              // P V of a tile retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 1);
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.H, b = blockIdx.x / p.H;
  int t0, t1;                                          // this CTA's key tiles (all of them with one split)
  x_split_tiles((p.Lk + kTile - 1) / kTile, gridDim.y, blockIdx.y, t0, t1);
  const int nt = t1 - t0;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kXStages; ++s) { mbar_init(k_full + s, 1); mbar_init(v_full + s, 1); mbar_init(kv_free + s, 1); }
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
    tma_load_4d_w(smem + S::OFF_Q, &tmQ, q_full, 0, 0, h, b);                 // rows >= nq: zero-filled
    for (int i = 0; i < nt; ++i) {
      const int s = i % kXStages;
      if (i >= kXStages) mbar_wait(kv_free + s, ((i / kXStages) - 1) & 1);
      mbar_arrive_expect_tx_w(k_full + s, S::TILE);
      tma_load_4d_w(smem + S::OFF_K + s * S::TILE, &tmK, k_full + s, 0, (t0 + i) * kTile, h, b);
      mbar_arrive_expect_tx_w(v_full + s, S::TILE);
      tma_load_4d_w(smem + S::OFF_V + s * S::TILE, &tmV, v_full + s, 0, (t0 + i) * kTile, h, b);
    }
  } else if (warp == 5) {
    // ---- MMA issuer: S(0); then per tile  S(i+1) ; wait P(i) ; O += P(i) V(i)   (in-order pipe: S(i+1) overwrites the
    //      buffer P(i-1) V(i-1) read only after that MMA)
    const uint32_t idesc_s = make_idesc(kTile, kTile, Elem<T>::fmt, 0, 0);
    const uint32_t idesc_pv = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
    const uint32_t q_addr = smem_u32(smem + S::OFF_Q);
    auto issue_s = [&](int i) {
      const int s = i % kXStages;
      mbar_wait(k_full + s, (i / kXStages) & 1);
      tc_fence_after();
      const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * S::TILE);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks)
        mma_ss_w(tmem_base + 128 * (i & 1), make_smem_desc(q_addr + ks * 32, 16, 8 * ROWB, ROWB),
                 make_smem_desc(k_addr + ks * 32, 16, 8 * ROWB, ROWB), idesc_s, ks > 0 ? 1u : 0u);
      tc_commit_w(s_ready + (i & 1));
    };
    mbar_wait(q_full, 0);
    issue_s(0);
    for (int i = 0; i < nt; ++i) {
      if (i + 1 < nt) issue_s(i + 1);
      const int s = i % kXStages;
      mbar_wait(p_ready + (i & 1), (i >> 1) & 1);
      mbar_wait(v_full + s, (i / kXStages) & 1);
      tc_fence_after();
      const uint32_t v_addr = smem_u32(smem + S::OFF_V + s * S::TILE);
#pragma unroll
      for (int k2 = 0; k2 < kTile / 16; ++k2)          // 16 keys per MMA: A = P (16-bit, 8 columns), B = V rows MN-major
        mma_ts_w(tmem_base + COL_O, tmem_base + 128 * (i & 1) + 8 * k2,
                 make_smem_desc(v_addr + k2 * 16 * ROWB, S::TILE, 8 * ROWB, ROWB), idesc_pv, (i > 0 || k2 > 0) ? 1u : 0u);
      tc_commit_w(o_done);
      tc_commit_w(kv_free + s);
    }
  } else {
    // ---- softmax / epilogue warps: warp w owns query rows 32 w .. 32 w + 31
    const int row = warp * 32 + lane;
    const bool warp_valid = warp * 32 < p.nq;            // warps without a valid query only keep the barriers going
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    float m = -INFINITY, l = 0.f;                        // running maximum (log2 domain) and row sum relative to it
    for (int i = 0; i < nt; ++i) {
      float* kp = sKpm + (i & 1) * kTile;
      {   // additive key terms of this tile: mask * log2(e), -inf beyond the sequence
        const int key = (t0 + i) * kTile + (int)threadIdx.x;
        float kv = -INFINITY;
        if (key < p.Lk) kv = p.kpm ? p.kpm[(int64_t)b * p.Lk + key] * kLog2e : 0.f;
        kp[threadIdx.x] = kv;
      }
      named_bar_sync(1, 128);
      mbar_wait(s_ready + (i & 1), (i >> 1) & 1);
      tc_fence_after();
      const uint32_t ts = trow + 128 * (i & 1);
      if (warp_valid) {
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
            tmax = fmaxf(tmax, fmaf(__uint_as_float(v[4 * e + 0]), p.scale_log2, kk.x));
            tmax = fmaxf(tmax, fmaf(__uint_as_float(v[4 * e + 1]), p.scale_log2, kk.y));
            tmax = fmaxf(tmax, fmaf(__uint_as_float(v[4 * e + 2]), p.scale_log2, kk.z));
            tmax = fmaxf(tmax, fmaf(__uint_as_float(v[4 * e + 3]), p.scale_log2, kk.w));
          }
        }
        float alpha = 1.f;
        if (tmax > m + kXRescale || m == -INFINITY) {    // (also the first tile and rows that were fully masked so far)
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
            const float p0 = fast_exp2(fmaf(__uint_as_float(v[4 * e + 0]), p.scale_log2, kk.x) + neg_m);
            const float p1 = fast_exp2(fmaf(__uint_as_float(v[4 * e + 1]), p.scale_log2, kk.y) + neg_m);
            const float p2 = fast_exp2(fmaf(__uint_as_float(v[4 * e + 2]), p.scale_log2, kk.z) + neg_m);
            const float p3 = fast_exp2(fmaf(__uint_as_float(v[4 * e + 3]), p.scale_log2, kk.w) + neg_m);
            l0 += p0 + p2;
            l1 += p1 + p3;
            pk[2 * e] = Elem<T>::pack(p0, p1);
            pk[2 * e + 1] = Elem<T>::pack(p2, p3);
          }
          tmem_st16(ts + 16 * c, pk);
        }
        l += l0 + l1;
        // lazy rescaling of the accumulator: O holds sums relative to the OLD maximum
        const bool any = __any_sync(0xffffffffu, alpha != 1.f);
        if (any && i > 0) {
          mbar_wait(o_done, (i - 1) & 1);               // P V of the previous tile has retired
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
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_ready + (i & 1));
    }
    mbar_wait(o_done, (nt - 1) & 1);
    tc_fence_after();
    if (gridDim.y > 1) {
      // epilogue of one split of several: O_s / l_s in fp32 and (m_s, l_s) for the merge launch.  A split whose keys are
      // all -inf has l_s = 0: its O_s is written as 0 and the merge gives it weight 0.
      const float inv = l > 0.f ? 1.0f / l : 0.f;
      const int64_t slot = ((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * p.nq + row;
#pragma unroll
      for (int half = 0; half < DH / 32; ++half) {
        uint32_t o[32];
        tmem_ld32(trow + COL_O + 32 * half, o);
        tmem_wait_ld(o);
        if (row < p.nq) {
          float4* dst = reinterpret_cast<float4*>(p.part_o + slot * DH + 32 * half);
#pragma unroll
          for (int e = 0; e < 8; ++e)
            dst[e] = make_float4(__uint_as_float(o[4 * e]) * inv, __uint_as_float(o[4 * e + 1]) * inv,
                                 __uint_as_float(o[4 * e + 2]) * inv, __uint_as_float(o[4 * e + 3]) * inv);
        }
      }
      if (row < p.nq) { p.part_m[slot] = m; p.part_l[slot] = l; }
    } else {
      // epilogue: O / l -> 16-bit -> swizzled staging (the Q tile) -> TMA store ; LSE
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
          *reinterpret_cast<uint4*>(stage + swz_off<ROWB>(row, half * 4 + cq)) = w4;
        }
      }
      if (row < p.nq) p.lse[((int64_t)b * p.H + h) * p.nq + row] = (m + log2f(l)) * kLn2;
      fence_proxy_async();
      named_bar_sync(1, 128);
      if (threadIdx.x == 0) {
        tma_store_4d(&tmO, stage, 0, 0, h, b);             // rows >= nq are outside the tensor: clipped
        tma_store_commit();
        tma_store_wait_all();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem_base);
}

// grid (B * H, nq), DH threads (one per output column): per (pair, query row), over the splits in order,  M = max_s m_s,  w_s = l_s 2^(m_s - M),
// out = sum_s w_s O_s / sum_s w_s,  lse = (M + log2 sum_s w_s) ln 2.  The split's (m_s, l_s) rather than its own lse
// travel to the merge: next to the -1e7 key mask an fp32 lse is a number near -1e7 whose spacing is 1, so a split's
// weight exp(lse_s - max lse) would be off by up to e^0.5, while m_s - M is exact there.
template <typename T, int DH>
__global__ void __launch_bounds__(DH)
xattn_fwd_merge_kernel(const float* __restrict__ part_o, const float* __restrict__ part_m, const float* __restrict__ part_l,
                       T* __restrict__ out, float* __restrict__ lse, int64_t os0, int64_t os1, int64_t os2, int H, int nq,
                       int splits) {
  const int pair = blockIdx.x, row = blockIdx.y, c = threadIdx.x, b = pair / H, h = pair - b * H;
  const int64_t base = (int64_t)pair * splits;
  float M = -INFINITY;
  for (int s = 0; s < splits; ++s) M = fmaxf(M, part_m[(base + s) * nq + row]);
  float L = 0.f, O = 0.f;
  for (int s = 0; s < splits; ++s) {
    const int64_t slot = (base + s) * nq + row;
    const float ms = part_m[slot];
    const float w = ms == -INFINITY ? 0.f : part_l[slot] * exp2f(ms - M);         // splits without a finite key: 0
    L += w;
    O = fmaf(w, part_o[slot * DH + c], O);
  }
  out[b * os0 + h * os1 + row * os2 + c] = from_f32<T>(O / L);     // no finite key at all: 0 / 0, as with one split
  if (c == 0) lse[(int64_t)pair * nq + row] = (M + log2f(L)) * kLn2;
}

bool xattn_supported(const svae_xattn_desc* d) {
  if (d->dtype != SVAE_DTYPE_BF16 && d->dtype != SVAE_DTYPE_F16) return false;
  return d->head_dim == 64 && d->num_queries >= 1 && d->num_queries <= 128 && d->num_keys >= 1 && d->scale > 0.f;
}

int xattn_key_tiles(const svae_xattn_desc* d) { return (d->num_keys + kTile - 1) / kTile; }

// The library's key split count.  One CTA per (batch, head) pair streams all keys of the pair; from kXMinPairs pairs on
// that fills the GPU well enough (and those shapes keep exactly the one-split launch).  Below it each pair gets about
// SMs / pairs CTAs (both kernels hold 512 TMEM columns: one CTA per SM, one wave), but every split keeps at least
// kXMinSplitTiles key tiles.  Measured on a B200 (1000 W, 148 SMs) at 16 x 4096 tokens, 8 heads: the forward takes 66 us
// with one split (32 tiles per CTA), 116 us with 16 (2 tiles per CTA) and 168 us with 32 -- a CTA's fixed work (TMEM
// allocation, Q load, pipeline fill, epilogue) costs about two tiles, so splits shorter than ~8 tiles mostly pay for it.
constexpr int kXMinPairs = 64;
constexpr int kXMinSplitTiles = 8;

int xattn_key_splits(const svae_xattn_desc* d) {
  const int64_t pairs = (int64_t)d->batch * d->heads;
  if (pairs <= 0 || pairs >= kXMinPairs) return 1;
  const int64_t want = sm_count_of_current_device() / pairs;
  return (int)std::max<int64_t>(1, std::min<int64_t>(want, xattn_key_tiles(d) / kXMinSplitTiles));
}

// fp32 partials: the forward's O_s, m_s, l_s; the backward's dQ_s (smaller) fits the same workspace
size_t xattn_workspace_bytes(const svae_xattn_desc* d, int splits) {
  if (splits <= 1) return 0;
  return sizeof(float) * (size_t)d->batch * d->heads * splits * d->num_queries * (d->head_dim + 2);
}

template <typename T>
static int launch_xattn_fwd(const svae_xattn_desc* d, int splits, const void* q, const void* k, const void* v, const float* kpm,
                            void* out, float* lse, float* ws, cudaStream_t st) {
  constexpr int DH = 64;
  using S = XFwdSmem<DH>;
  CUtensorMap tmQ, tmK, tmV, tmO;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  if ((rc = encode_tmap(&tmQ, dt, q, DH, d->num_queries, d->heads, d->batch, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, DH, d->num_keys, d->heads, d->batch, d->k_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, DH, d->num_keys, d->heads, d->batch, d->v_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmO, dt, out, DH, d->num_queries, d->heads, d->batch, d->o_stride, kTile))) return rc;
  const int pairs = d->batch * d->heads;
  const size_t parts = (size_t)pairs * splits * d->num_queries;
  XParams p;
  p.kpm = kpm; p.lse = lse; p.delta = nullptr;
  p.part_o = splits > 1 ? ws : nullptr;
  p.part_m = splits > 1 ? ws + parts * DH : nullptr;
  p.part_l = splits > 1 ? ws + parts * (DH + 1) : nullptr;
  p.nq = d->num_queries; p.Lk = d->num_keys; p.H = d->heads;
  p.scale = d->scale; p.scale_log2 = d->scale * kLog2e;
  auto kern = xattn_fwd_sm100_kernel<T, DH>;
  SVAE_CONFIGURE_SMEM(kern, S::DYN_BYTES);
  {
    ScopedKernelTimer timer("xattn_fwd_sm100", st);
    kern<<<dim3(pairs, splits), kXThreads, S::DYN_BYTES, st>>>(tmQ, tmK, tmV, tmO, p);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  if (splits > 1) {
    ScopedKernelTimer timer("xattn_fwd_merge", st);
    xattn_fwd_merge_kernel<T, DH><<<dim3(pairs, d->num_queries), DH, 0, st>>>(
        p.part_o, p.part_m, p.part_l, reinterpret_cast<T*>(out), lse, d->o_stride[0], d->o_stride[1], d->o_stride[2], d->heads,
        d->num_queries, splits);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  return SVAE_OK;
}

int xattn_fwd(const svae_xattn_desc* d, int splits, const void* q, const void* k, const void* v, const float* kpm, void* out,
              float* lse, float* ws, cudaStream_t st) {
  return d->dtype == SVAE_DTYPE_BF16 ? launch_xattn_fwd<__nv_bfloat16>(d, splits, q, k, v, kpm, out, lse, ws, st)
                                     : launch_xattn_fwd<__half>(d, splits, q, k, v, kpm, out, lse, ws, st);
}


// ------------------------------------------------------------------------------------------ backward
constexpr int kXBThreads = 512;

template <int DH>
struct XBwdSmem {
  static constexpr int ROWB = DH * 2;
  static constexpr int TILE = kTile * ROWB;
  static constexpr int OFF_K = 0;                                 // [kXStages] K tile, later the dK staging tile
  static constexpr int OFF_V = OFF_K + kXStages * TILE;           // [kXStages] V tile, later the dV staging tile
  static constexpr int OFF_Q = OFF_V + kXStages * TILE;           // Q (rows >= nq zero)
  static constexpr int OFF_DO = OFF_Q + TILE;                     // dO
  static constexpr int OFF_DS = OFF_DO + TILE;                    // dS^T [128 keys][64 queries] + a second, all-zero half
  static constexpr int OFF_STAT = OFF_DS + 2 * TILE;              // [2][128]: -lse*log2e, -delta*scale per query
  static constexpr int OFF_BAR = OFF_STAT + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int COL_U = 0, COL_DK = 256, COL_DV = 320, COL_DQ = 384;
};

struct XBwdParams {
  const float* kpm;
  const float* lse;
  const void *out, *dout;       // read directly for delta = rowsum(dO o O)
  void* dq;
  float* part_dq;               // key_splits > 1: [B*H][splits][nq][DH] the split's dQ_s, fp32
  int64_t o_stride[3], do_stride[3], dq_stride[3];
  int nq, Lk, H;
  float scale, scale_log2;
};

template <typename T, int DH>
__global__ void __launch_bounds__(kXBThreads, 1)
xattn_bwd_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                       const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                       const __grid_constant__ CUtensorMap tmDK, const __grid_constant__ CUtensorMap tmDV, const XBwdParams p) {
  static_assert(DH == 64, "128-byte rows");
  using S = XBwdSmem<DH>;
  constexpr int ROWB = S::ROWB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* k_full = bars + 0;        // [3]
  uint64_t* v_full = bars + 3;        // [3]
  uint64_t* kv_free = bars + 6;       // [3] epilogue: the stage's staging stores have been read
  uint64_t* q_full = bars + 9;        // Q and dO tiles
  uint64_t* s_ready = bars + 10;      // [2] per math group
  uint64_t* p_ready = bars + 12;      // [2] (one arrival per warp)
  uint64_t* u_free = bars + 14;       // [2] the group's TMEM operands have been consumed
  uint64_t* acc_ready = bars + 16;    // dK / dV of the tile (and dQ so far) retired
  uint64_t* acc_free = bars + 17;     // epilogue has read dK / dV (one arrival per warp)
  uint64_t* ds_free = bars + 18;      // the dQ MMAs have read the dS^T staging tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 19);
  float* sStat = reinterpret_cast<float*>(smem + S::OFF_STAT);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.H, b = blockIdx.x / p.H;
  int t0, t1;                                          // this CTA's key tiles (all of them with one split)
  x_split_tiles((p.Lk + kTile - 1) / kTile, gridDim.y, blockIdx.y, t0, t1);
  const int nt = t1 - t0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kXStages; ++s) { mbar_init(k_full + s, 1); mbar_init(v_full + s, 1); mbar_init(kv_free + s, 1); }
    mbar_init(q_full, 1);
    for (int k = 0; k < 2; ++k) { mbar_init(s_ready + k, 1); mbar_init(p_ready + k, 4); mbar_init(u_free + k, 1); }
    mbar_init(acc_ready, 1); mbar_init(acc_free, 4); mbar_init(ds_free, 1);
    fence_barrier_init();
  }
  if (warp == 15) {
    if (lane == 0) {
      prefetch_tensormap(&tmQ); prefetch_tensormap(&tmDO); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV);
      prefetch_tensormap(&tmDK); prefetch_tensormap(&tmDV);
    }
    tmem_alloc<512>(tmem_slot);
  }
  // the all-zero second half of the dS^T operand (queries 64..127 of the M = 128 MMA do not exist)
  for (int i = threadIdx.x; i < S::TILE / 16; i += kXBThreads)
    reinterpret_cast<uint4*>(smem + S::OFF_DS + S::TILE)[i] = make_uint4(0, 0, 0, 0);
  // statistics of the (<= 128) queries: -lse*log2e and -delta*scale, delta = rowsum(dO o O) straight from global memory;
  // queries that do not exist get -inf / 0 so that their P and dS columns come out as exact zeros
  if (threadIdx.x < kTile) {
    const int qi = threadIdx.x;
    float nl = -INFINITY, nd = 0.f;
    if (qi < p.nq) {
      const T* o = reinterpret_cast<const T*>(p.out) + b * p.o_stride[0] + h * p.o_stride[1] + qi * p.o_stride[2];
      const T* d_o = reinterpret_cast<const T*>(p.dout) + b * p.do_stride[0] + h * p.do_stride[1] + qi * p.do_stride[2];
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
      nl = -p.lse[((int64_t)b * p.H + h) * p.nq + qi] * kLog2e;
      nd = -d * p.scale;
    }
    sStat[qi] = nl;
    sStat[kTile + qi] = nd;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 12) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 12) {
      // ---- TMA producer
      mbar_arrive_expect_tx_w(q_full, 2 * S::TILE);
      tma_load_4d_w(smem + S::OFF_Q, &tmQ, q_full, 0, 0, h, b);
      tma_load_4d_w(smem + S::OFF_DO, &tmDO, q_full, 0, 0, h, b);
      for (int i = 0; i < nt; ++i) {
        const int s = i % kXStages;
        if (i >= kXStages) mbar_wait(kv_free + s, ((i / kXStages) - 1) & 1);
        mbar_arrive_expect_tx_w(k_full + s, S::TILE);
        tma_load_4d_w(smem + S::OFF_K + s * S::TILE, &tmK, k_full + s, 0, (t0 + i) * kTile, h, b);
        mbar_arrive_expect_tx_w(v_full + s, S::TILE);
        tma_load_4d_w(smem + S::OFF_V + s * S::TILE, &tmV, v_full + s, 0, (t0 + i) * kTile, h, b);
      }
    } else if (warp == 13) {
      // ---- S^T = K Q^T and dP^T = V dO^T (128 keys x 64 queries) into the score buffer of group i & 1
      const uint32_t idesc_s = make_idesc(kTile, 64, Elem<T>::fmt, 0, 0);
      const uint32_t q_addr = smem_u32(smem + S::OFF_Q), do_addr = smem_u32(smem + S::OFF_DO);
      mbar_wait(q_full, 0);
      for (int i = 0; i < nt; ++i) {
        const int s = i % kXStages, w = i & 1;
        mbar_wait(k_full + s, (i / kXStages) & 1);
        mbar_wait(v_full + s, (i / kXStages) & 1);
        if (i >= 2) mbar_wait(u_free + w, ((i >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * S::TILE), v_addr = smem_u32(smem + S::OFF_V + s * S::TILE);
        const uint32_t d_s = tmem_base + S::COL_U + 128 * w;
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks) {
          mma_ss_w(d_s, make_smem_desc(k_addr + ks * 32, 16, 8 * ROWB, ROWB), make_smem_desc(q_addr + ks * 32, 16, 8 * ROWB, ROWB),
                   idesc_s, ks > 0 ? 1u : 0u);
          mma_ss_w(d_s + 64, make_smem_desc(v_addr + ks * 32, 16, 8 * ROWB, ROWB), make_smem_desc(do_addr + ks * 32, 16, 8 * ROWB, ROWB),
                   idesc_s, ks > 0 ? 1u : 0u);
        }
        tc_commit_w(s_ready + w);
      }
    } else if (warp == 14) {
      // ---- dV = P^T dO, dK = dS^T Q (A from TMEM), dQ += dS K (A = staged dS^T read MN-major)
      const uint32_t idesc_o = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
      const uint32_t idesc_mn = make_idesc(kTile, DH, Elem<T>::fmt, 1, 1);
      const uint32_t q_addr = smem_u32(smem + S::OFF_Q), do_addr = smem_u32(smem + S::OFF_DO), ds_addr = smem_u32(smem + S::OFF_DS);
      for (int i = 0; i < nt; ++i) {
        const int s = i % kXStages, w = i & 1;
        mbar_wait(p_ready + w, (i >> 1) & 1);
        if (i >= 1) mbar_wait(acc_free, (i - 1) & 1);
        tc_fence_after();
        const uint32_t ta = tmem_base + S::COL_U + 128 * w;
        const uint32_t k_addr = smem_u32(smem + S::OFF_K + s * S::TILE);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {               // 16 queries per MMA
          mma_ts_w(tmem_base + S::COL_DV, ta + 8 * ks, make_smem_desc(do_addr + ks * 16 * ROWB, S::TILE, 8 * ROWB, ROWB), idesc_o,
                   ks > 0 ? 1u : 0u);
          mma_ts_w(tmem_base + S::COL_DK, ta + 64 + 8 * ks, make_smem_desc(q_addr + ks * 16 * ROWB, S::TILE, 8 * ROWB, ROWB), idesc_o,
                   ks > 0 ? 1u : 0u);
        }
#pragma unroll
        for (int k2 = 0; k2 < kTile / 16; ++k2)        // 16 keys per MMA
          mma_ss_w(tmem_base + S::COL_DQ, make_smem_desc(ds_addr + k2 * 16 * 128, S::TILE, 8 * 128, 128),
                   make_smem_desc(k_addr + k2 * 16 * ROWB, S::TILE, 8 * ROWB, ROWB), idesc_mn, (i > 0 || k2 > 0) ? 1u : 0u);
        tc_commit_w(u_free + w);                       // (after the dQ MMAs on purpose: see the math groups' ds_free wait)
        tc_commit_w(ds_free);
        tc_commit_w(acc_ready);
      }
    }
  } else if (warp >= 8) {
    // ---- epilogue group: dK, dV of every tile -> 16-bit -> the tile's own K / V buffers -> TMA store; dQ at the end
    asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
    const int w = warp & 3;
    const int tid_g = threadIdx.x & 127;
    const int row = w * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(w * 32) << 16);
    for (int i = 0; i < nt; ++i) {
      const int s = i % kXStages;
      mbar_wait(acc_ready, i & 1);
      tc_fence_after();
      uint8_t* stage[2] = {smem + S::OFF_K + s * S::TILE, smem + S::OFF_V + s * S::TILE};
#pragma unroll
      for (int which = 0; which < 2; ++which) {
#pragma unroll
        for (int half = 0; half < DH / 32; ++half) {
          uint32_t v[32];
          tmem_ld32(trow + (which ? S::COL_DV : S::COL_DK) + 32 * half, v);
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
      }
      tc_fence_before();
      mbar_arrive_warp(acc_free);
      fence_proxy_async();
      named_bar_sync(1, 128);
      if (tid_g == 0) {
        tma_store_4d(&tmDK, stage[0], 0, (t0 + i) * kTile, h, b);  // rows beyond Lk are outside the tensor: clipped
        tma_store_4d(&tmDV, stage[1], 0, (t0 + i) * kTile, h, b);
        tma_store_commit();
        tma_store_wait_read();
        mbar_arrive(kv_free + s);
      }
    }
    // dQ (complete after the last tile's MMAs): rows < nq, written directly -- or, as one split of several, drained in
    // fp32 for the reduce launch.  tcgen05.ld is warp-collective: every lane of a warp that owns at least one query takes
    // part in the loads, only the rows that exist are stored.
    if (gridDim.y > 1) {
      if (w * 32 < p.nq) {
        float* part = p.part_dq + (((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * p.nq + row) * DH;
#pragma unroll
        for (int half = 0; half < DH / 32; ++half) {
          uint32_t v[32];
          tmem_ld32(trow + S::COL_DQ + 32 * half, v);
          tmem_wait_ld(v);
          if (row < p.nq) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
              reinterpret_cast<float4*>(part)[half * 8 + e] = make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]),
                                                                           __uint_as_float(v[4 * e + 2]), __uint_as_float(v[4 * e + 3]));
          }
        }
      }
    } else if (w * 32 < p.nq) {
      T* dq = reinterpret_cast<T*>(p.dq) + b * p.dq_stride[0] + h * p.dq_stride[1] + row * p.dq_stride[2];
#pragma unroll
      for (int half = 0; half < DH / 32; ++half) {
        uint32_t v[32];
        tmem_ld32(trow + S::COL_DQ + 32 * half, v);
        tmem_wait_ld(v);
        if (row < p.nq) {
#pragma unroll
          for (int cq = 0; cq < 4; ++cq) {
            uint4 o;
            o.x = Elem<T>::pack(__uint_as_float(v[cq * 8 + 0]), __uint_as_float(v[cq * 8 + 1]));
            o.y = Elem<T>::pack(__uint_as_float(v[cq * 8 + 2]), __uint_as_float(v[cq * 8 + 3]));
            o.z = Elem<T>::pack(__uint_as_float(v[cq * 8 + 4]), __uint_as_float(v[cq * 8 + 5]));
            o.w = Elem<T>::pack(__uint_as_float(v[cq * 8 + 6]), __uint_as_float(v[cq * 8 + 7]));
            reinterpret_cast<uint4*>(dq)[half * 4 + cq] = o;
          }
        }
      }
    }
    if (tid_g == 0) tma_store_wait_all();
  } else {
    // ---- math groups: group i & 1 owns tile i; lane = key, 64 query columns in two halves of 32
    asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    const int wg = warp >> 2, c = warp & 3;
    const int row = c * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(c * 32) << 16);
    uint8_t* sDS = smem + S::OFF_DS;
    for (int i = wg; i < nt; i += 2) {
      const int key = (t0 + i) * kTile + row;
      float kv = -INFINITY;                              // additive key term (log2 domain); -inf beyond the sequence
      if (key < p.Lk) kv = p.kpm ? p.kpm[(int64_t)b * p.Lk + key] * kLog2e : 0.f;
      const uint32_t tb = trow + S::COL_U + 128 * wg;
      mbar_wait(s_ready + wg, (i >> 1) & 1);
      tc_fence_after();
      uint32_t dsr[32];                                  // the key's 64 dS values, 16-bit pairs
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t sv[32], dv[32], pk[16];
        tmem_ld32(tb + 32 * half, sv);
        tmem_ld32(tb + 64 + 32 * half, dv);
        tmem_wait_ld(sv, dv);
        const float4* nl = reinterpret_cast<const float4*>(sStat + 32 * half);
        const float4* nd = reinterpret_cast<const float4*>(sStat + kTile + 32 * half);
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
          const float4 l4 = nl[q4], d4 = nd[q4];
          const float lq[4] = {l4.x, l4.y, l4.z, l4.w}, dq[4] = {d4.x, d4.y, d4.z, d4.w};
          float pp[4], dd[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int qi = q4 * 4 + e;
            const float pe = fast_exp2(fmaf(__uint_as_float(sv[qi]), p.scale_log2, lq[e]) + kv);
            pp[e] = pe;
            dd[e] = pe * fmaf(__uint_as_float(dv[qi]), p.scale, dq[e]);
          }
          pk[q4 * 2] = Elem<T>::pack(pp[0], pp[1]);
          pk[q4 * 2 + 1] = Elem<T>::pack(pp[2], pp[3]);
          dsr[16 * half + q4 * 2] = Elem<T>::pack(dd[0], dd[1]);
          dsr[16 * half + q4 * 2 + 1] = Elem<T>::pack(dd[2], dd[3]);
        }
        // in place: P^T over the first 32 score columns, dS^T over the first 32 dP columns (all consumed by now:
        // half 1 overwrites columns 16..31 / 80..95, which half 0 has read)
        tmem_st16(tb + 16 * half, pk);
        uint32_t dsh[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) dsh[e] = dsr[16 * half + e];
        tmem_st16(tb + 64 + 16 * half, dsh);
      }
      // the previous tile's dQ MMAs have read the staging tile.  (The parity wait is unambiguous: this tile's scores
      // exist only because the group's buffer was released AFTER the dQ MMAs of tile i - 2, so that phase is complete.)
      if (i >= 1) mbar_wait(ds_free, (i - 1) & 1);
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)
        *reinterpret_cast<uint4*>(sDS + swz_off<128>(row, ch)) = make_uint4(dsr[4 * ch], dsr[4 * ch + 1], dsr[4 * ch + 2], dsr[4 * ch + 3]);
      fence_proxy_async();
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive_warp(p_ready + wg);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 15) tmem_dealloc<512>(tmem_base);
}

// grid (B * H, nq), DH threads: dq = sum_s dQ_s over the splits in order, rounded once to 16 bits
template <typename T, int DH>
__global__ void __launch_bounds__(DH)
xattn_dq_reduce_kernel(const float* __restrict__ part_dq, T* __restrict__ dq, int64_t s0, int64_t s1, int64_t s2, int H, int nq,
                       int splits) {
  const int pair = blockIdx.x, row = blockIdx.y, c = threadIdx.x, b = pair / H, h = pair - b * H;
  const int64_t base = (int64_t)pair * splits;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += part_dq[((base + s) * nq + row) * DH + c];
  dq[b * s0 + h * s1 + row * s2 + c] = from_f32<T>(acc);
}

template <typename T>
static int launch_xattn_bwd(const svae_xattn_desc* d, int splits, const void* q, const void* k, const void* v, const void* out,
                            const void* dout, const float* lse, const float* kpm, void* dq, void* dk, void* dv, float* ws,
                            cudaStream_t st) {
  constexpr int DH = 64;
  using S = XBwdSmem<DH>;
  CUtensorMap tmQ, tmDO, tmK, tmV, tmDK, tmDV;
  int rc;
  const CUtensorMapDataType dt = Elem<T>::tm;
  if ((rc = encode_tmap(&tmQ, dt, q, DH, d->num_queries, d->heads, d->batch, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmDO, dt, dout, DH, d->num_queries, d->heads, d->batch, d->do_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, dt, k, DH, d->num_keys, d->heads, d->batch, d->k_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmV, dt, v, DH, d->num_keys, d->heads, d->batch, d->v_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmDK, dt, dk, DH, d->num_keys, d->heads, d->batch, d->dk_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmDV, dt, dv, DH, d->num_keys, d->heads, d->batch, d->dv_stride, kTile))) return rc;
  XBwdParams p;
  p.kpm = kpm; p.lse = lse; p.out = out; p.dout = dout; p.dq = dq;
  p.part_dq = splits > 1 ? ws : nullptr;
  for (int i = 0; i < 3; ++i) { p.o_stride[i] = d->o_stride[i]; p.do_stride[i] = d->do_stride[i]; p.dq_stride[i] = d->dq_stride[i]; }
  p.nq = d->num_queries; p.Lk = d->num_keys; p.H = d->heads;
  p.scale = d->scale; p.scale_log2 = d->scale * kLog2e;
  auto kern = xattn_bwd_sm100_kernel<T, DH>;
  SVAE_CONFIGURE_SMEM(kern, S::DYN_BYTES);
  const int pairs = d->batch * d->heads;
  {
    ScopedKernelTimer timer("xattn_bwd_sm100", st);
    kern<<<dim3(pairs, splits), kXBThreads, S::DYN_BYTES, st>>>(tmQ, tmDO, tmK, tmV, tmDK, tmDV, p);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  if (splits > 1) {
    ScopedKernelTimer timer("xattn_bwd_dq_reduce", st);
    xattn_dq_reduce_kernel<T, DH><<<dim3(pairs, d->num_queries), DH, 0, st>>>(
        ws, reinterpret_cast<T*>(dq), d->dq_stride[0], d->dq_stride[1], d->dq_stride[2], d->heads, d->num_queries, splits);
    SVAE_CUDA_CHECK(cudaGetLastError());
  }
  return SVAE_OK;
}

int xattn_bwd(const svae_xattn_desc* d, int splits, const void* q, const void* k, const void* v, const void* out, const void* dout,
              const float* lse, const float* kpm, void* dq, void* dk, void* dv, float* ws, cudaStream_t st) {
  return d->dtype == SVAE_DTYPE_BF16 ? launch_xattn_bwd<__nv_bfloat16>(d, splits, q, k, v, out, dout, lse, kpm, dq, dk, dv, ws, st)
                                     : launch_xattn_bwd<__half>(d, splits, q, k, v, out, dout, lse, kpm, dq, dk, dv, ws, st);
}

}  // namespace sm100
}  // namespace svae

using namespace svae;

static bool x_tma_ok(const void* p, const int64_t s[3]) {
  return reinterpret_cast<uintptr_t>(p) % 16 == 0 && (s[0] * 2) % 16 == 0 && (s[1] * 2) % 16 == 0 && (s[2] * 2) % 16 == 0;
}

extern "C" int svae_xattn_supported(const svae_xattn_desc* d) { return d && sm100::xattn_supported(d) ? 1 : 0; }

// the checks of the forward / backward entries; `name` is the entry that reports a failure
static int x_check_fwd(const char* name, const svae_xattn_desc* d, const void* q, const void* k, const void* v, const void* out,
                       const float* lse) {
  SVAE_REQUIRE(d && q && k && v && out && lse, SVAE_ERR_INVALID, "%s: null argument", name);
  SVAE_REQUIRE(sm100::xattn_supported(d), SVAE_ERR_UNSUPPORTED,
               "%s: needs 16-bit tensors, head_dim 64 and 1..128 queries (got dtype %d, head_dim %d, %d queries)", name, d->dtype,
               d->head_dim, d->num_queries);
  SVAE_REQUIRE(x_tma_ok(q, d->q_stride) && x_tma_ok(k, d->k_stride) && x_tma_ok(v, d->v_stride) && x_tma_ok(out, d->o_stride),
               SVAE_ERR_INVALID, "%s: tensors must be 16-byte aligned with strides that are multiples of 8 elements", name);
  return SVAE_OK;
}

static int x_check_bwd(const char* name, const svae_xattn_desc* d, const void* q, const void* k, const void* v, const void* out,
                       const void* dout, const float* lse, const void* dq, const void* dk, const void* dv) {
  SVAE_REQUIRE(d && q && k && v && out && dout && lse && dq && dk && dv, SVAE_ERR_INVALID, "%s: null argument", name);
  SVAE_REQUIRE(sm100::xattn_supported(d), SVAE_ERR_UNSUPPORTED, "%s: needs 16-bit tensors, head_dim 64 and 1..128 queries", name);
  SVAE_REQUIRE(d->num_queries <= 64, SVAE_ERR_UNSUPPORTED, "%s: at most 64 queries (got %d)", name, d->num_queries);
  SVAE_REQUIRE(x_tma_ok(q, d->q_stride) && x_tma_ok(k, d->k_stride) && x_tma_ok(v, d->v_stride) && x_tma_ok(out, d->o_stride) &&
                   x_tma_ok(dout, d->do_stride) && x_tma_ok(dq, d->dq_stride) && x_tma_ok(dk, d->dk_stride) && x_tma_ok(dv, d->dv_stride),
               SVAE_ERR_INVALID, "%s: tensors must be 16-byte aligned with strides that are multiples of 8 elements", name);
  return SVAE_OK;
}

// key_splits within 1..key tiles and a workspace of svae_xattn_workspace_bytes (none needed for one split)
static int x_check_split(const char* name, const svae_xattn_desc* d, int key_splits, const void* ws, size_t ws_bytes) {
  const int tiles = sm100::xattn_key_tiles(d);
  SVAE_REQUIRE(key_splits >= 1 && key_splits <= tiles, SVAE_ERR_INVALID, "%s: key_splits %d outside 1..%d (the 128-key tiles of %d keys)",
               name, key_splits, tiles, d->num_keys);
  const size_t need = sm100::xattn_workspace_bytes(d, key_splits);
  SVAE_REQUIRE(need == 0 || (ws && ws_bytes >= need), SVAE_ERR_INVALID, "%s: workspace of %zu bytes at %p, %zu needed for %d key splits",
               name, ws_bytes, ws, need, key_splits);
  SVAE_REQUIRE(reinterpret_cast<uintptr_t>(ws) % 16 == 0, SVAE_ERR_INVALID, "%s: workspace must be 16-byte aligned", name);
  return SVAE_OK;
}

extern "C" int svae_xattn_key_splits(const svae_xattn_desc* d) {
  SVAE_REQUIRE(d && sm100::xattn_supported(d) && d->batch > 0 && d->heads > 0, SVAE_ERR_INVALID,
               "svae_xattn_key_splits: null or unsupported descriptor");
  return sm100::xattn_key_splits(d);
}

extern "C" size_t svae_xattn_workspace_bytes(const svae_xattn_desc* d, int key_splits) {
  if (!d || !sm100::xattn_supported(d) || key_splits < 1 || key_splits > sm100::xattn_key_tiles(d)) return 0;
  return sm100::xattn_workspace_bytes(d, key_splits);
}

extern "C" int svae_xattn_fwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v,
                              const float* key_padding_mask, void* out, float* lse, void* stream) {
  int rc;
  if ((rc = x_check_fwd("svae_xattn_fwd", d, q, k, v, out, lse))) return rc;
  return sm100::xattn_fwd(d, 1, q, k, v, key_padding_mask, out, lse, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int svae_xattn_fwd_split(const svae_xattn_desc* d, int key_splits, const void* q, const void* k, const void* v,
                                    const float* key_padding_mask, void* out, float* lse, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  int rc;
  if ((rc = x_check_fwd("svae_xattn_fwd_split", d, q, k, v, out, lse))) return rc;
  if ((rc = x_check_split("svae_xattn_fwd_split", d, key_splits, workspace, workspace_bytes))) return rc;
  return sm100::xattn_fwd(d, key_splits, q, k, v, key_padding_mask, out, lse, static_cast<float*>(workspace),
                          static_cast<cudaStream_t>(stream));
}

extern "C" int svae_xattn_bwd(const svae_xattn_desc* d, const void* q, const void* k, const void* v, const void* out,
                              const void* dout, const float* lse, const float* key_padding_mask, void* dq, void* dk, void* dv,
                              void* stream) {
  int rc;
  if ((rc = x_check_bwd("svae_xattn_bwd", d, q, k, v, out, dout, lse, dq, dk, dv))) return rc;
  return sm100::xattn_bwd(d, 1, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int svae_xattn_bwd_split(const svae_xattn_desc* d, int key_splits, const void* q, const void* k, const void* v,
                                    const void* out, const void* dout, const float* lse, const float* key_padding_mask, void* dq,
                                    void* dk, void* dv, void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = x_check_bwd("svae_xattn_bwd_split", d, q, k, v, out, dout, lse, dq, dk, dv))) return rc;
  if ((rc = x_check_split("svae_xattn_bwd_split", d, key_splits, workspace, workspace_bytes))) return rc;
  return sm100::xattn_bwd(d, key_splits, q, k, v, out, dout, lse, key_padding_mask, dq, dk, dv, static_cast<float*>(workspace),
                          static_cast<cudaStream_t>(stream));
}
