// Persistent, warp-specialised fused block-sparse attention forward (sm_100a) for the reference's default geometry
// (<= 8 key slots per 128-query tile, <= 4 live band blocks per block-row).
//
// One CTA per SM walks over query tiles (tile = blockIdx.x + i * gridDim.x), two tiles in TMEM at any time and a
// third in its epilogue, 16 warps:
//   warps 0-3   softmax group 0 (tiles 0, 2, ...)  | one batch of tcgen05.ld of the block-row's live slots, two-pass
//   warps 4-7   softmax group 1 (tiles 1, 3, ...)  | register-resident softmax, P written over S in TMEM, LSE
//   warps 8-11  epilogue group (every tile): (O_even + O_odd) / l -> 16-bit -> swizzled SMEM -> TMA store; frees TMEM
//   warp 12     TMA producer: Q + K (2-deep ring, refilled when the tile's S = Q K^T MMAs retire) and V (2-deep ring,
//               refilled when both P V chains retire)
//   warp 13     tcgen05.mma issuer: S(i) = Q K^T (never blocks on another tile's softmax)
//   warp 14/15  tcgen05.mma issuers: the even- / odd-slot half of O(i) = P V
// TMEM: 2 x 256 columns (per tile: S 256 | P aliases 0-127 | O_even 128-191 | O_odd 192-255).  Registers are
// rebalanced with setmaxnreg (softmax 184, epilogue 88, producers 40).  While group 0 runs the CUDA-core softmax of
// tile i, group 1 works on tile i+1, the epilogue group drains tile i-1, the tensor pipe computes the next S and the
// TMA engine is already fetching tile i+2.  Same arithmetic as attn_fwd_sm100_kernel.
#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kPersistThreads = 512;

template <int DH>
struct FwdPSmem {
  static constexpr int NS = 8;
  static constexpr int ROWB = DH * 2;
  static constexpr int Q_BYTES = kTile * ROWB;
  static constexpr int SLOT_BYTES = kBlock * ROWB;
  static constexpr int KV_BYTES = NS * SLOT_BYTES;
  static constexpr int OFF_Q = 0;                            // [2]
  static constexpr int OFF_K = OFF_Q + 2 * Q_BYTES;          // [2]
  static constexpr int OFF_V = OFF_K + 2 * KV_BYTES;         // [2]
  static constexpr int OFF_OST = OFF_V + 2 * KV_BYTES;       // [2] output staging
  static constexpr int OFF_KPM = OFF_OST + 2 * Q_BYTES;      // [2]
  static constexpr int OFF_INV = OFF_KPM + 2 * NS * kBlock * 4;   // [2][128] 1 / row sum, softmax -> epilogue
  static constexpr int OFF_BAR = OFF_INV + 2 * kTile * 4;
  static constexpr int DYN_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int O_COL = 128, O2_COL = 192;
  static_assert(DYN_BYTES <= 227 * 1024, "shared memory");
};

template <typename T, int DH>
__global__ void __launch_bounds__(kPersistThreads, 1)
attn_fwd_persist_sm100_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                              const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmKband,
                              const __grid_constant__ CUtensorMap tmVband, const __grid_constant__ CUtensorMap tmO,
                              const FwdParams p, const int tiles_per_seq, const int num_tiles) {
  using S = FwdPSmem<DH>;
  constexpr int ROWB = S::ROWB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* qk_full = bars + 0;     // [2] TMA -> MMA
  uint64_t* v_full = bars + 2;      // [2] TMA -> the two P V issuers
  uint64_t* qk_free = bars + 4;     // [2] S retired -> Q/K producer
  uint64_t* v_free = bars + 6;      // [2] both P V chains retired -> V producer              (2 arrivals)
  uint64_t* s_ready = bars + 8;     // [2] MMA -> softmax group
  uint64_t* p_ready = bars + 10;    // [2] softmax group -> the two P V issuers                (128 arrivals)
  uint64_t* o_ready = bars + 12;    // [2] both P V chains retired -> epilogue group           (2 arrivals)
  uint64_t* tmem_free = bars + 14;  // [2] epilogue has read O: TMEM half reusable             (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const TileGeom g = p.g;
  const int ns = g.nslots;
  const int nt = (num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;     // tiles of this CTA

  if (threadIdx.x == 0) {
    for (int k = 0; k < 2; ++k) {
      mbar_init(qk_full + k, 1); mbar_init(v_full + k, 1); mbar_init(qk_free + k, 1); mbar_init(v_free + k, 2);
      mbar_init(s_ready + k, 1); mbar_init(p_ready + k, 128); mbar_init(o_ready + k, 2); mbar_init(tmem_free + k, 128);
    }
    fence_barrier_init();
  }
  if (warp == 15) {
    if (lane == 0) {
      prefetch_tensormap(&tmQ); prefetch_tensormap(&tmK); prefetch_tensormap(&tmV);
      prefetch_tensormap(&tmKband); prefetch_tensormap(&tmVband); prefetch_tensormap(&tmO);
    }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto tile_coords = [&](int i, int& t, int& h, int& b) {
    const int id = (int)blockIdx.x + i * (int)gridDim.x;
    t = id % tiles_per_seq;
    const int bh = id / tiles_per_seq;
    h = bh % p.H;
    b = bh / p.H;
  };
  const uint32_t idesc_pv = make_idesc(kTile, DH, Elem<T>::fmt, 0, 1);
  // O (+)= P_j V_j for slots j = first, first + 2, ... of the tile in ring slot k
  auto issue_pv_chain = [&](int k, int first, uint32_t o_col) {
    const uint32_t v_addr = smem_u32(smem + S::OFF_V + k * S::KV_BYTES);
    const uint32_t tb = tmem_base + 256 * k;
    uint32_t acc = 0;
    for (int j = first; j < ns; j += 2) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const uint64_t bd = make_smem_desc(v_addr + j * S::SLOT_BYTES + s * 16 * ROWB, S::SLOT_BYTES, 8 * ROWB, ROWB);
        mma_ts_w(tb + o_col, tb + 16 * j + 8 * s, bd, idesc_pv, acc);
        acc = 1;
      }
    }
  };

  if (warp >= 12) {
    // ======================================= producers / MMA issuers ========================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 12) {
      // ---- TMA producer: Q + K of tile i as soon as S(i-2) has retired, V of tile i as soon as P V(i-2) has retired
      for (int i = 0; i < nt; ++i) {
        const int k = i & 1, n = i >> 1;
        int t, h, b;
        tile_coords(i, t, h, b);
        const int band_lo = 4 * t - (g.left - 1);
        if (i >= 2) mbar_wait(qk_free + k, (n - 1) & 1);
        uint8_t* sQ = smem + S::OFF_Q + k * S::Q_BYTES;
        uint8_t* sK = smem + S::OFF_K + k * S::KV_BYTES;
        mbar_arrive_expect_tx_w(qk_full + k, S::Q_BYTES + ns * S::SLOT_BYTES);
        tma_load_4d_w(sQ, &tmQ, qk_full + k, 0, t * kTile, h, b);
        tma_load_4d_w(sK + g.cls * S::SLOT_BYTES, &tmKband, qk_full + k, 0, band_lo * kBlock, h, b);   // OOB rows -> zeros
        if (g.cls) tma_load_4d_w(sK, &tmK, qk_full + k, 0, 0, h, b);
        if (i >= 2) mbar_wait(v_free + k, (n - 1) & 1);
        uint8_t* sV = smem + S::OFF_V + k * S::KV_BYTES;
        mbar_arrive_expect_tx_w(v_full + k, ns * S::SLOT_BYTES);
        tma_load_4d_w(sV + g.cls * S::SLOT_BYTES, &tmVband, v_full + k, 0, band_lo * kBlock, h, b);
        if (g.cls) tma_load_4d_w(sV, &tmV, v_full + k, 0, 0, h, b);
      }
    } else if (warp == 13) {
      // ---- S(i) = Q K^T into TMEM half k; never blocks on the softmax of another tile
      const uint32_t idesc_s = make_idesc(kTile, ns * kBlock, Elem<T>::fmt, 0, 0);
      for (int i = 0; i < nt; ++i) {
        const int k = i & 1, n = i >> 1;
        mbar_wait(qk_full + k, n & 1);
        if (i >= 2) mbar_wait(tmem_free + k, (n - 1) & 1);
        tc_fence_after();
        const uint32_t q_addr = smem_u32(smem + S::OFF_Q + k * S::Q_BYTES);
        const uint32_t k_addr = smem_u32(smem + S::OFF_K + k * S::KV_BYTES);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_ss_w(tmem_base + 256 * k, make_smem_desc(q_addr + ks * 32, 16, 8 * ROWB, ROWB),
                   make_smem_desc(k_addr + ks * 32, 16, 8 * ROWB, ROWB), idesc_s, ks > 0 ? 1u : 0u);
        tc_commit_w(s_ready + k);
        tc_commit_w(qk_free + k);
      }
    } else {
      // ---- warp 14: even-slot half of O(i) = P V, warp 15: odd-slot half
      const int first = warp - 14;
      for (int i = 0; i < nt; ++i) {
        const int k = i & 1, n = i >> 1;
        mbar_wait(p_ready + k, n & 1);
        mbar_wait(v_full + k, n & 1);
        tc_fence_after();
        issue_pv_chain(k, first, first ? S::O2_COL : S::O_COL);
        tc_commit_w(o_ready + k);
        tc_commit_w(v_free + k);
      }
    }
  } else if (warp >= 8) {
    // ======================================= epilogue group ==================================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
    const int w = warp & 3;                    // TMEM lane quarter
    const int tid_g = threadIdx.x & 127;
    const int row = w * 32 + lane;
    for (int i = 0; i < nt; ++i) {
      const int k = i & 1, n = i >> 1;
      int t, h, b;
      tile_coords(i, t, h, b);
      const uint32_t trow = tmem_base + 256 * k + ((uint32_t)(w * 32) << 16);
      uint8_t* sOst = smem + S::OFF_OST + k * S::Q_BYTES;
      const float* sInv = reinterpret_cast<const float*>(smem + S::OFF_INV) + k * kTile;
      mbar_wait(o_ready + k, n & 1);
      tc_fence_after();
      const float inv = sInv[row];             // written before the group's p_ready arrival (ordered through the MMA warp)
      uint32_t oa[32], ob[32];
      uint32_t pk[DH / 2];
#pragma unroll
      for (int half = 0; half < DH / 32; ++half) {
        tmem_ld32(trow + S::O_COL + 32 * half, oa);
        tmem_ld32(trow + S::O2_COL + 32 * half, ob);
        tmem_wait_ld(oa, ob);
        if (half == DH / 32 - 1) {
          tc_fence_before();
          mbar_arrive(tmem_free + k);          // S / P / O of this TMEM half are consumed
        }
#pragma unroll
        for (int c = 0; c < 32; c += 2)
          pk[half * 16 + (c >> 1)] = Elem<T>::pack((__uint_as_float(oa[c]) + __uint_as_float(ob[c])) * inv,
                                                   (__uint_as_float(oa[c + 1]) + __uint_as_float(ob[c + 1])) * inv);
      }
#pragma unroll
      for (int ch = 0; ch < DH / 8; ++ch)
        *reinterpret_cast<uint4*>(sOst + swz_off<ROWB>(row, ch)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
      fence_proxy_async();
      named_bar_sync(3, 128);
      if (tid_g == 0) {
        tma_store_4d(&tmO, sOst, 0, t * kTile, h, b);
        tma_store_commit();
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");    // the OTHER staging tile has been read
      }
      named_bar_sync(3, 128);                  // nobody writes the other staging tile before its store has read it
    }
    if (tid_g == 0) tma_store_wait_all();
  } else {
    // ======================================= softmax groups ==================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 184;");
    const int grp = warp >> 2;                 // 0 or 1 = ring slot / TMEM half of this group's tiles
    const int w = warp & 3;                    // TMEM lane quarter = block-row inside the tile
    const int tid_g = threadIdx.x & 127;
    const int row = w * 32 + lane;
    const uint32_t tb = tmem_base + 256 * grp;
    const uint32_t trow = tb + ((uint32_t)(w * 32) << 16);
    float* sKpm = reinterpret_cast<float*>(smem + S::OFF_KPM) + grp * (S::NS * kBlock);
    float* sInv = reinterpret_cast<float*>(smem + S::OFF_INV) + grp * kTile;
    const uint32_t below_diag = (lane == 31) ? 0xffffffffu : ((2u << lane) - 1u);   // bit c set <=> key c <= query lane
    const int nlb = g.left + g.nsup;           // live band slots per block-row (<= 4)
    const int first = g.cls + w;
    const int kdiag = g.causal ? g.left - 1 : -1;

    for (int i = grp; i < nt; i += 2) {
      const int n = i >> 1;
      int t, h, b;
      tile_coords(i, t, h, b);
      const int r0 = 4 * t, r = r0 + w;
      const int band_lo = r0 - (g.left - 1);
      const int qpos = t * kTile + row;
      auto slot_valid = [&](int j) {
        if (g.cls && j == 0) return true;
        int blk = band_lo + j - g.cls;
        return blk >= g.cls && blk < g.nb;
      };

      // stage the additive key-padding mask of the tile's keys (log2 domain); all-zero -> fast path
      uint32_t any_kpm = 0;
      if (p.kpm) {
        for (int e = tid_g; e < ns * kBlock; e += 128) {
          const int j = e >> 5, c = e & 31;
          float kv = 0.f;
          if (slot_valid(j)) {
            const int blk = (g.cls && j == 0) ? 0 : band_lo + j - g.cls;
            kv = p.kpm[(int64_t)b * p.L + blk * kBlock + c] * kLog2e;
          }
          sKpm[e] = kv;
          any_kpm |= (kv != 0.f) ? 1u : 0u;
        }
      }
      const bool has_kpm = p.kpm ? bar_red_or(1 + grp, 128, any_kpm) : false;

      const bool lg = g.cls && r < g.nb;
      bool lv[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) lv[kk] = kk < nlb && r < g.nb && slot_valid(first + kk);

      mbar_wait(s_ready + grp, n & 1);
      tc_fence_after();
      // Both passes are ROLLED loops over the block-row's live slots (k = 0: global block, k = 1..4: band slot
      // first + k - 1), re-reading the scores from TMEM in pass 2: tcgen05.ld is cheap (~53 cycles per 4 KB per SMSP,
      // profiles/r01b_pipe_bench.log) while ~1.5 k instructions of straight-line code per tile do not fit the instruction
      // cache next to the other warps' streams (13 % `no_inst` stalls in profiles/r01b_persist_hot_sass.txt).
      float m = -INFINITY, l0 = 0.f, l1 = 0.f;
      const bool g_diag = g.causal && g.cls && r == 0 && lg;      // block-row 0: the global block IS the diagonal
      uint32_t live_bits = lg ? 1u : 0u;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) live_bits |= lv[kk] ? (2u << kk) : 0u;
      // ---- pass 1: row maximum
#pragma unroll 1
      for (int k = 0; k < 5; ++k) {
        if (!((live_bits >> k) & 1u)) continue;
        const int j = k == 0 ? 0 : first + k - 1;
        uint32_t v[32];
        tmem_ld32(trow + 32 * j, v);
        tmem_wait_ld(v);
        if (k == 0 ? g_diag : (kdiag == k - 1)) mask_above_diag(v, below_diag);
        m = slot_max(v, m, has_kpm, sKpm + j * kBlock, p.scale_log2);
      }
      if (!has_kpm) m *= p.scale_log2;        // scale > 0: max commutes with the scaling
      const float neg_m = (m == -INFINITY) ? 0.f : -m;

      // ---- pass 2: P = exp2(s * scale_log2 + mask - m), written over S as packed 16-bit.  Slots are visited in
      //      increasing column order, so P_j (columns 16 j ..) only ever overwrites scores that were already consumed.
      uint32_t pk[16];
#pragma unroll 1
      for (int k = 0; k < 5; ++k) {
        if (!((live_bits >> k) & 1u)) continue;
        const int j = k == 0 ? 0 : first + k - 1;
        uint32_t v[32];
        tmem_ld32(trow + 32 * j, v);
        tmem_wait_ld(v);
        if (k == 0 ? g_diag : (kdiag == k - 1)) mask_above_diag(v, below_diag);
        slot_exp_pack<T>(v, pk, l0, l1, has_kpm, sKpm + j * kBlock, p.scale_log2, neg_m);
        tmem_st16(trow + 16 * j, pk);
      }
#pragma unroll
      for (int c = 0; c < 16; ++c) pk[c] = 0u;
      uint32_t live_mask = lg ? 1u : 0u;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) live_mask |= lv[kk] ? (1u << (first + kk)) : 0u;
      for (int j = 0; j < ns; ++j)              // P = 0 for the slots this block-row does not attend
        if (!((live_mask >> j) & 1u)) tmem_st16(trow + 16 * j, pk);
      const float l = l0 + l1;
      sInv[row] = 1.0f / l;                     // l == 0 (row with every key masked) -> inf * 0 = NaN, like the reference softmax
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_ready + grp);
      if (qpos < p.L) p.lse[((int64_t)b * p.H + h) * p.L + qpos] = (m + log2f(l)) * kLn2;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 15) tmem_dealloc<512>(tmem_base);
}

template <typename T, int DH>
static int launch_fwd_persist(const svae_attn_desc* d, const TileGeom& g, const void* q, const void* k, const void* v,
                              const float* kpm, void* out, float* lse, cudaStream_t st) {
  using S = FwdPSmem<DH>;
  CUtensorMap tmQ, tmK, tmV, tmKb, tmVb, tmO;
  int rc;
  const int band_rows = g.nband * kBlock;
  if ((rc = encode_tmap(&tmQ, Elem<T>::tm, q, DH, d->seq_len, d->heads, d->batch, d->q_stride, kTile))) return rc;
  if ((rc = encode_tmap(&tmK, Elem<T>::tm, k, DH, d->seq_len, d->heads, d->batch, d->k_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmV, Elem<T>::tm, v, DH, d->seq_len, d->heads, d->batch, d->v_stride, kBlock))) return rc;
  if ((rc = encode_tmap(&tmKb, Elem<T>::tm, k, DH, d->seq_len, d->heads, d->batch, d->k_stride, band_rows))) return rc;
  if ((rc = encode_tmap(&tmVb, Elem<T>::tm, v, DH, d->seq_len, d->heads, d->batch, d->v_stride, band_rows))) return rc;
  if ((rc = encode_tmap(&tmO, Elem<T>::tm, out, DH, d->seq_len, d->heads, d->batch, d->o_stride, kTile))) return rc;
  FwdParams p;
  p.kpm = kpm; p.lse = lse; p.s_dump = nullptr;
  p.L = d->seq_len; p.H = d->heads; p.g = g;
  p.scale_log2 = d->scale * kLog2e;
  auto kern = attn_fwd_persist_sm100_kernel<T, DH>;
  const int sm_count = sm_count_of_current_device();
  SVAE_CONFIGURE_SMEM(kern, S::DYN_BYTES);
  const int tiles_per_seq = (d->seq_len + kTile - 1) / kTile;
  const int num_tiles = tiles_per_seq * d->heads * d->batch;
  const int grid = num_tiles < sm_count ? num_tiles : sm_count;
  ScopedKernelTimer timer("attn_fwd_sm100", st);
  kern<<<grid, kPersistThreads, S::DYN_BYTES, st>>>(tmQ, tmK, tmV, tmKb, tmVb, tmO, p, tiles_per_seq, num_tiles);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

bool fwd_persist_supported(const svae_attn_desc* d) {
  if (d->dtype != SVAE_DTYPE_BF16 && d->dtype != SVAE_DTYPE_F16) return false;
  if (d->head_dim != 64 && d->head_dim != 32) return false;
  const TileGeom g = make_geom(d->window_size, d->causal, d->include_cls, d->seq_len / d->block_size);
  return g.nslots <= 8 && g.left + g.nsup <= 4 && d->scale > 0.f;
}

int fwd_persist(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out,
                float* lse, cudaStream_t st) {
  const TileGeom g = make_geom(d->window_size, d->causal, d->include_cls, d->seq_len / d->block_size);
  if (d->dtype == SVAE_DTYPE_BF16)
    return d->head_dim == 64 ? launch_fwd_persist<__nv_bfloat16, 64>(d, g, q, k, v, kpm, out, lse, st)
                             : launch_fwd_persist<__nv_bfloat16, 32>(d, g, q, k, v, kpm, out, lse, st);
  return d->head_dim == 64 ? launch_fwd_persist<__half, 64>(d, g, q, k, v, kpm, out, lse, st)
                           : launch_fwd_persist<__half, 32>(d, g, q, k, v, kpm, out, lse, st);
}

}  // namespace sm100
}  // namespace svae
