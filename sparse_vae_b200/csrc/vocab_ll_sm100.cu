// Per-token log-likelihood under the vocabulary head, without the logits (reference core/continuous_autoencoder.py:62-88
// `estimate_log_prob_iw` -> p_of_x_given_z: log_softmax(output_layer(hidden))[..., label], column 0 zeroed after the
// softmax).  One GEMM h @ W^T whose epilogue keeps a running log-sum-exp per row:
//   logit[r, c] = round16(sum_k h[r, k] w[c, k] + bias[c])         fp32 accumulation in TMEM, rounded like cuBLAS
//   logp[r]     = logit[r, label[r]] - logsumexp_c logit[r, c]     fp32; 0 where label[r] == 0
// The [rows, vocab] logits never leave the SM: h and W are read, 4 bytes per row are written.
//
// One persistent CTA per SM walks over 128-row tiles (tile = blockIdx.x + i * gridDim.x), 10 warps:
//   warp 8      TMA producer: the tile's h (d / 64 SWIZZLE_128B slices of 128 x 64, kept for the whole tile) and a
//               ring of W stages (256 vocabulary rows x 64 K-elements = 32 KB each)
//   warp 9      tcgen05.mma issuer (128 x 256 x 16, kind::f16): vocabulary tile j into TMEM accumulator j & 1
//   warps 0-7   epilogue: warp w reads TMEM lane quarter w & 3, columns (w >> 2) * 128 .. + 127 of each accumulator,
//               rounds to 16 bit, and updates an online max / sum of exponentials per row; the two column halves of
//               a row are combined in a fixed order at the end of the tile (deterministic, no atomics).
// TMEM: 2 x 256 columns, so the epilogue of vocabulary tile j overlaps the MMAs of tile j + 1.
#include "attn_sm100.cuh"

namespace svae {
namespace sm100 {

using namespace ptx;

constexpr int kVlThreads = 320;
constexpr int kVlN = 256;                          // vocabulary columns per MMA / TMEM accumulator
constexpr int kVlHSlice = kTile * 128;             // one 128-row x 64-element slice of h (16 KB)
constexpr int kVlWStage = kVlN * 128;              // one 256-row x 64-element slice of W (32 KB)
constexpr int kVlMaxStages = 8;
constexpr int kVlAux = 2048;                       // barriers, TMEM address, [3][128] floats of the half-combine
constexpr int kVlSmemLimit = 227 * 1024;

struct VlLayout {
  int ks, stages, bytes;
};
static VlLayout vl_layout(int d) {
  VlLayout l;
  l.ks = d / 64;
  const int free_bytes = kVlSmemLimit - 1024 - kVlAux - l.ks * kVlHSlice;
  l.stages = free_bytes / kVlWStage < kVlMaxStages ? free_bytes / kVlWStage : kVlMaxStages;
  l.bytes = l.ks * kVlHSlice + l.stages * kVlWStage + kVlAux + 1024;
  return l;
}

struct VlParams {
  const int64_t* labels;
  float* logp;
  const void* bias;
  int64_t rows;
  int vocab, ks, stages, num_tiles;
};

template <typename T> __device__ __forceinline__ uint32_t hmax2(uint32_t a, uint32_t b);
template <> __device__ __forceinline__ uint32_t hmax2<__nv_bfloat16>(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
template <> __device__ __forceinline__ uint32_t hmax2<__half>(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

// e == o ? a : b, opaque to the compiler: a select chain over a register array written with plain C++ is turned into
// an indexed load from a local-memory copy of the array
__device__ __forceinline__ uint32_t select_eq(int e, int o, uint32_t a, uint32_t b) {
  uint32_t r;
  asm("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %1, %2;\n\tselp.b32 %0, %3, %4, p;\n\t}" : "=r"(r) : "r"(e), "r"(o), "r"(a), "r"(b));
  return r;
}

// 32 accumulator columns (fp32 bits) + bias -> 16 packed pairs of 16-bit logits
template <typename T, bool BIAS>
__device__ __forceinline__ void round_logits(const uint32_t (&v)[32], const T* bias, uint32_t* pk) {
  uint4 braw[4];
  if (BIAS) {
#pragma unroll
    for (int q = 0; q < 4; ++q) braw[q] = __ldg(reinterpret_cast<const uint4*>(bias) + q);
  }
#pragma unroll
  for (int e = 0; e < 16; ++e) {
    float2 x = make_float2(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1]));
    if (BIAS) {
      const uint4 b4 = braw[e >> 2];
      const uint32_t bw = (e & 3) == 0 ? b4.x : (e & 3) == 1 ? b4.y : (e & 3) == 2 ? b4.z : b4.w;
      x = fadd2(x, Elem<T>::unpack(bw));
    }
    pk[e] = Elem<T>::pack(x.x, x.y);
  }
}

template <typename T, bool BIAS>
__global__ void __launch_bounds__(kVlThreads, 1)
vocab_logprob_sm100_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmW, const VlParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int KS = p.ks, NST = p.stages, NV = p.vocab / kVlN;
  uint8_t* sH = smem;
  uint8_t* sW = smem + KS * kVlHSlice;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sW + NST * kVlWStage);
  uint64_t* h_full = bars + 0;         // TMA -> MMA: the tile's h is in shared memory
  uint64_t* h_free = bars + 1;         // MMA -> TMA: every MMA reading h has retired
  uint64_t* acc_full = bars + 2;       // [2] MMA -> epilogue
  uint64_t* acc_free = bars + 4;       // [2] epilogue -> MMA (8 warp arrivals)
  uint64_t* w_full = bars + 6;         // [kVlMaxStages] TMA -> MMA
  uint64_t* w_free = bars + 6 + kVlMaxStages;   // [kVlMaxStages] MMA -> TMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6 + 2 * kVlMaxStages);
  float* part = reinterpret_cast<float*>(bars + 8 + 2 * kVlMaxStages);    // [3][128]

  const int warp = warp_index(), lane = threadIdx.x & 31;
  const int nt = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (threadIdx.x == 0) {
    mbar_init(h_full, 1);
    mbar_init(h_free, 1);
    for (int k = 0; k < 2; ++k) { mbar_init(acc_full + k, 1); mbar_init(acc_free + k, 8); }
    for (int s = 0; s < NST; ++s) { mbar_init(w_full + s, 1); mbar_init(w_free + s, 1); }
    fence_barrier_init();
  }
  if (warp == 9) {
    if (lane == 0) { prefetch_tensormap(&tmH); prefetch_tensormap(&tmW); }
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 8) {
    // ================================ TMA producer ================================
    uint32_t st = 0;
    for (int i = 0; i < nt; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      if (i > 0) mbar_wait(h_free, (i - 1) & 1);
      mbar_arrive_expect_tx_w(h_full, KS * kVlHSlice);
      for (int ks = 0; ks < KS; ++ks) tma_load_2d_w(sH + ks * kVlHSlice, &tmH, h_full, ks * 64, tile * kTile);
      for (int j = 0; j < NV; ++j) {
        for (int ks = 0; ks < KS; ++ks, ++st) {
          const uint32_t s = st % NST, u = st / NST;
          if (u > 0) mbar_wait(w_free + s, (u - 1) & 1);
          mbar_arrive_expect_tx_w(w_full + s, kVlWStage);
          tma_load_2d_w(sW + s * kVlWStage, &tmW, w_full + s, ks * 64, j * kVlN);
        }
      }
    }
  } else if (warp == 9) {
    // ================================ MMA issuer ==================================
    const uint32_t idesc = make_idesc(kTile, kVlN, Elem<T>::fmt, 0, 0);
    uint32_t st = 0, g = 0;
    for (int i = 0; i < nt; ++i) {
      mbar_wait(h_full, i & 1);
      tc_fence_after();
      for (int j = 0; j < NV; ++j, ++g) {
        const uint32_t k = g & 1;
        if (g >= 2) mbar_wait(acc_free + k, ((g >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + kVlN * k;
        for (int ks = 0; ks < KS; ++ks, ++st) {
          const uint32_t s = st % NST;
          mbar_wait(w_full + s, (st / NST) & 1);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sH + ks * kVlHSlice), b_addr = smem_u32(sW + s * kVlWStage);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_ss_w(d_tmem, make_smem_desc(a_addr + kk * 32, 16, 1024, 128), make_smem_desc(b_addr + kk * 32, 16, 1024, 128),
                     idesc, (ks | kk) != 0 ? 1u : 0u);
          tc_commit_w(w_free + s);
        }
        tc_commit_w(acc_full + k);
      }
      tc_commit_w(h_free);
    }
  } else {
    // ================================ epilogue ====================================
    constexpr float kL2e = kLog2e;
    const int q = warp & 3, half = warp >> 2;
    const int r_in = q * 32 + lane;
    const T* bias = reinterpret_cast<const T*>(p.bias);
    uint32_t g = 0;
    for (int i = 0; i < nt; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      const int64_t row = (int64_t)tile * kTile + r_in;
      const int64_t label = row < p.rows ? p.labels[row] : -1;
      float m = -INFINITY, x_label = 0.f;
      float2 sa = make_float2(0.f, 0.f), sb = make_float2(0.f, 0.f);
      for (int j = 0; j < NV; ++j, ++g) {
        const uint32_t k = g & 1;
        mbar_wait(acc_full + k, (g >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + kVlN * k + ((uint32_t)(q * 32) << 16) + half * 128;
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          const int col0 = j * kVlN + half * 128 + c * 64;
          uint32_t va[32], vb[32];
          tmem_ld32(taddr + 64 * c, va);
          tmem_ld32(taddr + 64 * c + 32, vb);
          tmem_wait_ld(va, vb);
          if (c == 1) {                      // both halves of the accumulator are in registers: TMEM reusable
            tc_fence_before();
            mbar_arrive_warp(acc_free + k);
          }
          uint32_t pk[32];
          round_logits<T, BIAS>(va, bias + col0, pk);
          round_logits<T, BIAS>(vb, bias + col0 + 32, pk + 16);
          // chunk maximum on the packed 16-bit values (exact), then one rescale of the running sum
          uint32_t mx = hmax2<T>(pk[0], pk[1]);
#pragma unroll
          for (int e = 2; e < 32; ++e) mx = hmax2<T>(mx, pk[e]);
          const float2 mf = Elem<T>::unpack(mx);
          const float m_new = fmaxf(m, fmaxf(mf.x, mf.y));
          const float scale = fast_exp2((m - m_new) * kL2e);      // m = -inf on the first chunk: 0 * 0
          sa = fmul2(sa, splat(scale));
          sb = fmul2(sb, splat(scale));
          m = m_new;
          const float nb = -m * kL2e;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float2 xa = ffma2(Elem<T>::unpack(pk[e]), splat(kL2e), splat(nb));
            const float2 xb = ffma2(Elem<T>::unpack(pk[e + 1]), splat(kL2e), splat(nb));
            sa = fadd2(sa, make_float2(fast_exp2(xa.x), fast_exp2(xa.y)));
            sb = fadd2(sb, make_float2(fast_exp2(xb.x), fast_exp2(xb.y)));
          }
          if (label >= col0 && label < col0 + 64) {                 // rare and divergent: pick the label's logit
            const int off = (int)(label - col0);
            uint32_t w = 0;
#pragma unroll
            for (int e = 0; e < 32; ++e) w = select_eq(e, off >> 1, pk[e], w);
            const float2 f = Elem<T>::unpack(w);
            x_label = (off & 1) ? f.y : f.x;
          }
        }
      }
      // combine the two column halves of each row in a fixed order: half 0 (this tile's columns 0-127) first
      const float s = (sa.x + sa.y) + (sb.x + sb.y);
      if (half == 1) {
        part[r_in] = m;
        part[128 + r_in] = s;
        part[256 + r_in] = x_label;
      }
      named_bar_sync(1, 256);
      if (half == 0 && row < p.rows) {
        const float m1 = part[r_in], s1 = part[128 + r_in], xl1 = part[256 + r_in];
        const float mm = fmaxf(m, m1);
        const float ss = s * fast_exp2((m - mm) * kL2e) + s1 * fast_exp2((m1 - mm) * kL2e);
        const float lse = mm + log2f(ss) * kLn2;
        p.logp[row] = label == 0 ? 0.f : (x_label + xl1) - lse;     // exactly one of the halves holds the label
      }
      named_bar_sync(1, 256);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc<512>(tmem_base);
}

template <typename T, bool BIAS>
static int launch_vocab_logprob(const void* h, int64_t ldh, const void* w, int64_t ldw, const void* bias, int64_t rows,
                                int vocab, int d, const int64_t* labels, float* logp, cudaStream_t st) {
  CUtensorMap tmH, tmW;
  int rc;
  if ((rc = encode_tmap_2d(&tmH, Elem<T>::tm, h, d, rows, ldh, kTile))) return rc;
  if ((rc = encode_tmap_2d(&tmW, Elem<T>::tm, w, d, vocab, ldw, kVlN))) return rc;
  const VlLayout l = vl_layout(d);
  VlParams p;
  p.labels = labels; p.logp = logp; p.bias = bias; p.rows = rows;
  p.vocab = vocab; p.ks = l.ks; p.stages = l.stages;
  p.num_tiles = (int)((rows + kTile - 1) / kTile);
  auto kern = vocab_logprob_sm100_kernel<T, BIAS>;
  SVAE_CONFIGURE_SMEM(kern, kVlSmemLimit);           // the largest layout (d = 512): one setting for every d
  const int sm_count = sm_count_of_current_device();
  const int grid = p.num_tiles < sm_count ? p.num_tiles : sm_count;
  ScopedKernelTimer timer("vocab_logprob_sm100", st);
  kern<<<grid, kVlThreads, l.bytes, st>>>(tmH, tmW, p);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

}  // namespace sm100
}  // namespace svae

using namespace svae;
using namespace svae::sm100;

extern "C" int svae_vocab_logprob_supported(int32_t vocab, int32_t d, int32_t dtype) {
  return (vocab >= kVlN && vocab % kVlN == 0 && d >= 64 && d <= 512 && d % 64 == 0 &&
          (dtype == SVAE_DTYPE_BF16 || dtype == SVAE_DTYPE_F16)) ? 1 : 0;
}

extern "C" int svae_vocab_logprob(const void* h, int64_t ldh, const void* w, int64_t ldw, const void* bias, int32_t dtype,
                                  int64_t rows, int32_t vocab, int32_t d, const int64_t* labels, float* logp, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SVAE_REQUIRE(h && w && labels && logp && rows >= 0, SVAE_ERR_INVALID, "svae_vocab_logprob: null argument");
  SVAE_REQUIRE(svae_vocab_logprob_supported(vocab, d, dtype), SVAE_ERR_UNSUPPORTED,
               "svae_vocab_logprob: vocab %d (256*k), d %d (64*k <= 512), dtype %d (16-bit) not supported", vocab, d, dtype);
  SVAE_REQUIRE(ldh >= d && ldw >= d && ldh % 8 == 0 && ldw % 8 == 0 && (reinterpret_cast<uintptr_t>(h) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0,
               SVAE_ERR_INVALID, "svae_vocab_logprob: h / w / bias must be 16-byte aligned with row strides of 8*k elements");
  SVAE_REQUIRE(rows < ((int64_t)1 << 31) - kTile, SVAE_ERR_INVALID, "svae_vocab_logprob: too many rows for one launch");
  if (rows == 0) return SVAE_OK;
  if (dtype == SVAE_DTYPE_BF16)
    return bias ? launch_vocab_logprob<__nv_bfloat16, true>(h, ldh, w, ldw, bias, rows, vocab, d, labels, logp, st)
                : launch_vocab_logprob<__nv_bfloat16, false>(h, ldh, w, ldw, bias, rows, vocab, d, labels, logp, st);
  return bias ? launch_vocab_logprob<__half, true>(h, ldh, w, ldw, bias, rows, vocab, d, labels, logp, st)
              : launch_vocab_logprob<__half, false>(h, ldh, w, ldw, bias, rows, vocab, d, labels, logp, st);
}
