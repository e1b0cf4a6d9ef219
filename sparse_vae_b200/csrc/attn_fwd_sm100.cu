// Fused block-sparse attention forward for sm_100a: TMA -> SMEM -> tcgen05.mma (S = Q K^T into TMEM) ->
// softmax on the TMEM rows (scale, additive key-padding, causal diagonal, band layout) -> P (16-bit) written back
// over S in TMEM -> tcgen05.mma (O = P V, A operand from TMEM) -> normalise -> swizzled SMEM -> TMA store.
// S and P never touch HBM (the reference materialises both: core/sparse_attention.py:84-92).
//
// One CTA = one 128-query tile (4 block-rows of the 32x32 layout) of one (batch, head).  The union of key blocks
// those 4 block-rows attend is a contiguous band of (left+3+nsup) blocks plus the global block 0, i.e. <= 8 "slots"
// of 32 keys at window 4; all of it fits TMEM at once (128 lanes x 32*slots fp32 columns).  Each of the 4 softmax
// warps owns exactly one block-row (TMEM lane quarter), so block sparsity is warp-uniform: a warp visits only its
// LIVE slots (<= 4 band + global at window 4) in two rolled passes (row maximum, then exp2 + pack), re-reading the
// scores from TMEM in the second pass, and dead blocks cost nothing on the CUDA cores.
// This is the one-CTA-per-tile variant: it serves the wide windows (9..14 slots, 512 TMEM columns) and the debug
// dumps; the default geometry runs the persistent kernel of attn_fwd_persist_sm100.cu (same arithmetic, bit for bit).
// TMEM budget: S [0, 32*slots) ; P aliases S ; two O accumulators in dead S columns (the P V chain is split over two
// issuing warps because one thread retires a TMEM-operand MMA only every ~123 cycles).  <= 256 columns -> two CTAs
// per SM overlap each other's load / MMA / softmax / store phases.  The whole band arrives with ONE TMA box per
// operand (rows outside [0, L) are zero-filled by the TMA unit).  All TMA / MMA issue is warp-convergent.
//
// Roofline: HBM-bound (AI ~ 79 FLOP/B at window 4, ridge ~ 215): algorithmic bytes = 4 * B*L*H*Dh * 2 per launch.
#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

template <int DH, int NSMAX>
struct FwdSmem {
  static constexpr int ROWB = DH * 2;
  static constexpr int Q_BYTES = kTile * ROWB;
  static constexpr int SLOT_BYTES = kBlock * ROWB;
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_K = OFF_Q + Q_BYTES;
  static constexpr int OFF_V = OFF_K + NSMAX * SLOT_BYTES;
  static constexpr int OFF_KPM = OFF_V + NSMAX * SLOT_BYTES;
  static constexpr int OFF_BAR = OFF_KPM + NSMAX * kBlock * 4;
  static constexpr int TOTAL = OFF_BAR + 64;
  static constexpr int DYN_BYTES = TOTAL + 1024;   // slack for manual 1024-byte alignment
  static constexpr bool kTwoChains = NSMAX <= 8;
  static constexpr int TMEM_COLS = NSMAX <= 8 ? 256 : 512;
  static constexpr int O_COL = NSMAX <= 8 ? 128 : 448;
  static constexpr int O2_COL = 192;               // second accumulator (two-chain variant only)
  static_assert(O_COL + DH <= TMEM_COLS, "O does not fit");
  static_assert(NSMAX * kBlock / 2 <= O_COL, "P must not overlap O");
};

template <typename T, int DH, int NSMAX>
__global__ void __launch_bounds__(kThreads, NSMAX <= 8 ? 2 : 1)
attn_fwd_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                      const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmKband,
                      const __grid_constant__ CUtensorMap tmVband, const __grid_constant__ CUtensorMap tmKband2,
                      const __grid_constant__ CUtensorMap tmVband2, const __grid_constant__ CUtensorMap tmO,
                      const FwdParams p) {
  using S = FwdSmem<DH, NSMAX>;
  constexpr int ROWB = S::ROWB;
  constexpr bool kTwoChains = S::kTwoChains;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem + S::OFF_Q;
  uint8_t* sK = smem + S::OFF_K;
  uint8_t* sV = smem + S::OFF_V;
  float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* bar_qk = bars + 0;   // TMA: Q + K slots landed
  uint64_t* bar_v = bars + 1;    // TMA: V slots landed
  uint64_t* bar_s = bars + 2;    // MMA: S complete in TMEM
  uint64_t* bar_p = bars + 3;    // softmax: P written to TMEM (128 arrivals)
  uint64_t* bar_o = bars + 4;    // MMA: O complete in TMEM (one arrival per P V chain)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const TileGeom g = p.g;
  const int ns = g.nslots;
  const int r0 = 4 * t;
  const int band_lo = r0 - (g.left - 1);

  auto slot_block = [&](int j) { return (g.cls && j == 0) ? 0 : band_lo + j - g.cls; };
  // a slot carries keys the tile may attend: inside the sequence and not a duplicate of the global block.
  // (every slot is LOADED -- out-of-range rows arrive as zeros -- so invalid slots only need P = 0)
  auto slot_valid = [&](int j) {
    if (g.cls && j == 0) return true;
    int blk = band_lo + j - g.cls;
    return blk >= g.cls && blk < g.nb;
  };

  if (threadIdx.x == 0) {
    mbar_init(bar_qk, 1);
    mbar_init(bar_v, 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, kTwoChains ? 2 : 1);
    fence_barrier_init();
  }
  if (warp == 4) {
    if (lane == 0) {
      prefetch_tensormap(&tmQ);
      prefetch_tensormap(&tmK);
      prefetch_tensormap(&tmV);
      prefetch_tensormap(&tmKband);
      prefetch_tensormap(&tmVband);
      prefetch_tensormap(&tmO);
    }
    tmem_alloc<S::TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const uint32_t v_addr = smem_u32(sV);
  const uint32_t idesc_pv = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
  // O (+)= P_j V_j for slots j = first, first + step, ... : A = P from TMEM (8 columns per 16 keys), B = V slot MN-major
  auto issue_pv_chain = [&](int first, int step, uint32_t o_col) {
    uint32_t acc = 0;
    for (int j = first; j < ns; j += step) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const uint64_t bd = make_smem_desc(v_addr + j * S::SLOT_BYTES + s * 16 * ROWB, S::SLOT_BYTES, 8 * ROWB, ROWB);
        mma_ts_w(tmem_base + o_col, tmem_base + 16 * j + 8 * s, bd, idesc_pv, acc);
        acc = 1;
      }
    }
  };

  if (warp == 4) {
    // ================= producer + MMA issuer: the whole warp runs this convergently, one lane is elected per op ====
    const int band_slots = ns - g.cls;
    mbar_arrive_expect_tx_w(bar_qk, S::Q_BYTES + ns * S::SLOT_BYTES);
    tma_load_4d_w(sQ, &tmQ, bar_qk, 0, t * kTile, h, b);
    tma_load_4d_w(sK + g.cls * S::SLOT_BYTES, &tmKband, bar_qk, 0, band_lo * kBlock, h, b);    // OOB rows -> zeros
    if (band_slots > 8) tma_load_4d_w(sK + (g.cls + 8) * S::SLOT_BYTES, &tmKband2, bar_qk, 0, (band_lo + 8) * kBlock, h, b);
    if (g.cls) tma_load_4d_w(sK, &tmK, bar_qk, 0, 0, h, b);
    mbar_arrive_expect_tx_w(bar_v, ns * S::SLOT_BYTES);
    tma_load_4d_w(sV + g.cls * S::SLOT_BYTES, &tmVband, bar_v, 0, band_lo * kBlock, h, b);
    if (band_slots > 8) tma_load_4d_w(sV + (g.cls + 8) * S::SLOT_BYTES, &tmVband2, bar_v, 0, (band_lo + 8) * kBlock, h, b);
    if (g.cls) tma_load_4d_w(sV, &tmV, bar_v, 0, 0, h, b);

    // ---- S = Q K^T : M = 128, N = 32*ns (split at 256), K = DH in steps of 16
    mbar_wait(bar_qk, 0);
    tc_fence_after();
    const uint32_t q_addr = smem_u32(sQ), k_addr = smem_u32(sK);
    const int ntot = ns * kBlock;
    for (int n0 = 0; n0 < ntot; n0 += 256) {
      const int n = (ntot - n0) < 256 ? (ntot - n0) : 256;
      const uint32_t idesc = make_idesc(kTile, n, Elem<T>::fmt, 0, 0);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        const uint64_t ad = make_smem_desc(q_addr + ks * 32, 16, 8 * ROWB, ROWB);
        const uint64_t bd = make_smem_desc(k_addr + n0 * ROWB + ks * 32, 16, 8 * ROWB, ROWB);
        mma_ss_w(tmem_base + n0, ad, bd, idesc, ks > 0 ? 1u : 0u);
      }
    }
    tc_commit_w(bar_s);

    // ---- O = P V, chain A (every second slot when a softmax warp issues the other half)
    mbar_wait(bar_p, 0);
    mbar_wait(bar_v, 0);
    tc_fence_after();
    issue_pv_chain(0, kTwoChains ? 2 : 1, S::O_COL);
    tc_commit_w(bar_o);
  } else {
    // ================= softmax + epilogue warps: warp w <-> block-row r0 + w <-> TMEM lanes 32w.. =================
    const int r = r0 + warp;
    const int row = warp * 32 + lane;
    const int qpos = t * kTile + row;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);

    // stage the additive key-padding mask (log2 domain); tiles whose keys are all unmasked take the fast path
    uint32_t any_kpm = 0;
    if (p.kpm) {
      for (int i = threadIdx.x; i < ns * kBlock; i += 128) {
        const int j = i >> 5, c = i & 31;
        float kv = 0.f;
        if (slot_valid(j)) kv = p.kpm[(int64_t)b * p.L + slot_block(j) * kBlock + c] * kLog2e;
        sKpm[i] = kv;
        any_kpm |= (kv != 0.f) ? 1u : 0u;
      }
    }
    const bool has_kpm = bar_red_or(1, 128, any_kpm);

    auto slot_live = [&](int j) {
      if (r >= g.nb || !slot_valid(j)) return false;
      if (g.cls && j == 0) return true;
      const int blk = band_lo + j - g.cls;
      return blk >= r - (g.left - 1) && blk <= r + g.nsup;
    };
    const uint32_t below_diag = (lane == 31) ? 0xffffffffu : ((2u << lane) - 1u);   // bit c set <=> key c <= query lane

    mbar_wait(bar_s, 0);
    tc_fence_after();

    if (p.s_dump) {   // debug only
      for (int j = 0; j < ns; ++j) {
        uint32_t v[32];
        tmem_ld32(trow + 32 * j, v);
        tmem_wait_ld(v);
        if (qpos < p.L) {
          float* dst = p.s_dump + (((int64_t)b * p.H + h) * p.L + qpos) * (ns * kBlock) + j * kBlock;
#pragma unroll
          for (int c = 0; c < 32; ++c) dst[c] = __uint_as_float(v[c]);
        }
      }
    }

    float m = -INFINITY, l0 = 0.f, l1 = 0.f, neg_m;
    {
      // ---- two ROLLED passes over the block-row's live slots, one TMEM round trip per slot and pass: tcgen05.ld is
      //      cheap (~53 cycles per 4 KB per SMSP) while straight-line code for 5 x 32 register-resident scores does not
      //      fit the instruction cache (measured on the persistent kernel: 92 -> 69 us, profiles/README.md)
      for (int j = 0; j < ns; ++j) {
        if (!slot_live(j)) continue;
        uint32_t v[32];
        tmem_ld32(trow + 32 * j, v);
        tmem_wait_ld(v);
        if (g.causal && slot_block(j) == r) mask_above_diag(v, below_diag);
        m = slot_max(v, m, has_kpm, sKpm + j * kBlock, p.scale_log2);
      }
      if (!has_kpm) m *= p.scale_log2;
      neg_m = (m == -INFINITY) ? 0.f : -m;
      for (int j = 0; j < ns; ++j) {
        uint32_t pk[16];
        if (slot_live(j)) {
          uint32_t v[32];
          tmem_ld32(trow + 32 * j, v);
          tmem_wait_ld(v);
          if (g.causal && slot_block(j) == r) mask_above_diag(v, below_diag);
          slot_exp_pack<T>(v, pk, l0, l1, has_kpm, sKpm + j * kBlock, p.scale_log2, neg_m);
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) pk[c] = 0u;
        }
        tmem_st16(trow + 16 * j, pk);     // in-order: only overwrites S columns that were already consumed
      }
    }
    const float l = l0 + l1;
    tmem_wait_st();
    tc_fence_before();
    mbar_arrive(bar_p);

    if (kTwoChains && warp == 0) {
      // ---- O2 = P V, chain B (odd slots), issued by this warp while it would otherwise idle until O is ready
      mbar_wait(bar_p, 0);
      mbar_wait(bar_v, 0);
      tc_fence_after();
      issue_pv_chain(1, 2, S::O2_COL);
      tc_commit_w(bar_o);
    }

    // ---- epilogue: (O + O2) / l -> 16-bit -> swizzled staging tile (reuses the Q buffer) -> TMA store ; LSE
    if (qpos < p.L) p.lse[((int64_t)b * p.H + h) * p.L + qpos] = (m + log2f(l)) * kLn2;
    const float inv = 1.0f / l;     // l == 0 (row with every key masked) -> NaN, like the reference softmax
    mbar_wait(bar_o, 0);
    tc_fence_after();
#pragma unroll
    for (int half = 0; half < DH / 32; ++half) {
      uint32_t v[32];
      tmem_ld32(trow + S::O_COL + 32 * half, v);
      if (kTwoChains) {
        uint32_t v2[32];
        tmem_ld32(trow + S::O2_COL + 32 * half, v2);
        tmem_wait_ld(v, v2);
#pragma unroll
        for (int c = 0; c < 32; ++c) v[c] = __float_as_uint(__uint_as_float(v[c]) + __uint_as_float(v2[c]));
      } else {
        tmem_wait_ld(v);
      }
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        uint4 w;
        w.x = Elem<T>::pack(__uint_as_float(v[cq * 8 + 0]) * inv, __uint_as_float(v[cq * 8 + 1]) * inv);
        w.y = Elem<T>::pack(__uint_as_float(v[cq * 8 + 2]) * inv, __uint_as_float(v[cq * 8 + 3]) * inv);
        w.z = Elem<T>::pack(__uint_as_float(v[cq * 8 + 4]) * inv, __uint_as_float(v[cq * 8 + 5]) * inv);
        w.w = Elem<T>::pack(__uint_as_float(v[cq * 8 + 6]) * inv, __uint_as_float(v[cq * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(sQ + swz_off<ROWB>(row, half * 4 + cq)) = w;
      }
    }
    fence_proxy_async();
    named_bar_sync(1, 128);
    if (threadIdx.x == 0) {
      tma_store_4d(&tmO, sQ, 0, t * kTile, h, b);
      tma_store_commit();
      tma_store_wait_read();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc<S::TMEM_COLS>(tmem_base);
}

template <typename T, int DH, int NSMAX>
static int launch_fwd(const svae_attn_desc* d, const TileGeom& g, const void* q, const void* k, const void* v,
                      const float* kpm, void* out, float* lse, float* s_dump, cudaStream_t st) {
  using S = FwdSmem<DH, NSMAX>;
  CUtensorMap tmQ, tmK, tmV, tmKb, tmVb, tmKb2, tmVb2, tmO;
  int rc;
  const int band_rows = (g.nband <= 8 ? g.nband : 8) * kBlock;
  const int band2_rows = (g.nband > 8 ? g.nband - 8 : 1) * kBlock;
  if ((rc = encode_tmap(&tmQ, Elem<T>::tm, q, DH, d->seq_len, d->heads, d->batch, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, Elem<T>::tm, k, DH, d->seq_len, d->heads, d->batch, d->k_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmV, Elem<T>::tm, v, DH, d->seq_len, d->heads, d->batch, d->v_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmKb, Elem<T>::tm, k, DH, d->seq_len, d->heads, d->batch, d->k_stride, band_rows))) return rc;
  if ((rc = encode_tmap(&tmVb, Elem<T>::tm, v, DH, d->seq_len, d->heads, d->batch, d->v_stride, band_rows))) return rc;
  if ((rc = encode_tmap(&tmKb2, Elem<T>::tm, k, DH, d->seq_len, d->heads, d->batch, d->k_stride, band2_rows))) return rc;
  if ((rc = encode_tmap(&tmVb2, Elem<T>::tm, v, DH, d->seq_len, d->heads, d->batch, d->v_stride, band2_rows))) return rc;
  if ((rc = encode_tmap(&tmO, Elem<T>::tm, out, DH, d->seq_len, d->heads, d->batch, d->o_stride, kTile))) return rc;
  FwdParams p;
  p.kpm = kpm; p.lse = lse; p.s_dump = s_dump;
  p.L = d->seq_len; p.H = d->heads; p.g = g;
  p.scale_log2 = d->scale * kLog2e;
  auto kern = attn_fwd_sm100_kernel<T, DH, NSMAX>;
  SVAE_CONFIGURE_SMEM(kern, S::DYN_BYTES);
  dim3 grid((d->seq_len + kTile - 1) / kTile, d->heads, d->batch);
  ScopedKernelTimer timer("attn_fwd_sm100", st);
  kern<<<grid, kThreads, S::DYN_BYTES, st>>>(tmQ, tmK, tmV, tmKb, tmVb, tmKb2, tmVb2, tmO, p);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

int fwd_max_slots() { return 14; }

int fwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out, float* lse,
        float* s_dump, cudaStream_t st) {
  const TileGeom g = make_geom(d->window_size, d->causal, d->include_cls, d->seq_len / d->block_size);
  SVAE_REQUIRE(g.nslots <= 14, SVAE_ERR_UNSUPPORTED, "sm100 attention forward: %d key slots (window %d) exceed 14",
               g.nslots, d->window_size);
  SVAE_REQUIRE(d->scale > 0.f, SVAE_ERR_UNSUPPORTED, "sm100 attention forward: softmax scale must be positive");
  const bool small = g.nslots <= 8 && g.left + g.nsup <= 4;   // the register-resident softmax holds <= 4 band slots
#define SVAE_FWD(T, DH)                                                                              \
  return small ? launch_fwd<T, DH, 8>(d, g, q, k, v, kpm, out, lse, s_dump, st)                      \
               : launch_fwd<T, DH, 14>(d, g, q, k, v, kpm, out, lse, s_dump, st)
  if (d->dtype == SVAE_DTYPE_BF16) {
    if (d->head_dim == 64) { SVAE_FWD(__nv_bfloat16, 64); }
    if (d->head_dim == 32) { SVAE_FWD(__nv_bfloat16, 32); }
  } else if (d->dtype == SVAE_DTYPE_F16) {
    if (d->head_dim == 64) { SVAE_FWD(__half, 64); }
    if (d->head_dim == 32) { SVAE_FWD(__half, 32); }
  }
#undef SVAE_FWD
  SVAE_REQUIRE(false, SVAE_ERR_UNSUPPORTED, "sm100 attention forward: dtype %d / head_dim %d not supported", d->dtype,
               d->head_dim);
}

}  // namespace sm100
}  // namespace svae
