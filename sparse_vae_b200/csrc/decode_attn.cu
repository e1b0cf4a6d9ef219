// Token-by-token decoding step of one sparse-attention layer (SURVEY.md section 8f row 3; reference
// core/attention.py:60-100 with the KV cache of :107-142, driven by TransformerVAE.sample, transformer_vae.py:112-126).
//
// The reference runs ~25 launches per layer and token: rotary on q and k (offset = cache_index), two cache row
// writes, a block shift of the cache every 32 tokens, q k^T, scale, softmax, p v.  Here it is ONE launch whose
// position comes from a device counter, so the whole per-token model step can sit in a CUDA graph:
//   * rotary (fp32 tables, one rounding to T -- the arithmetic of rotary.cu's autocast mode) on the new q and k rows,
//   * k / v appended to the cache.  Cache layout [B, (window+1)*block, d_model]: slots [0, block) hold positions
//     0..block-1 (the global block, never evicted), the other window*block slots are a RING over positions >= block
//     (position p lives in slot block + (p - block) mod (window*block)).  While p < (window+1)*block this is
//     the reference's layout (slot == p); afterwards the reference shifts the window left by one block every `block`
//     tokens where this kernel wraps around -- the set of visible keys is the same:
//     block 0 plus key blocks max(1, b - window + 1) .. b of the current block b (the rows of get_master_layout),
//   * scores, fp32 softmax and p v for every head of one sample.
// One CTA per (sample, head), one warp per 32 cache slots.  HBM-bound: reads the live part of both caches once,
// 2 * B * min(p+1, (window+1)*block) * d_model * sizeof(T) bytes per launch.
#include "common.cuh"

namespace svae {

template <typename T, int N> struct alignas(sizeof(T) * N) DPack { T v[N]; };

// position held by ring slot `slot` when the newest position is `pos`; -1 when the slot is empty or evicted
__device__ __forceinline__ int slot_position(int slot, int pos, int block, int window) {
  if (slot < block) return slot <= pos ? slot : -1;
  if (pos < block) return -1;
  const int ring = window * block;
  const int r = slot - block, m = pos - block;
  int back = (m - r) % ring;
  if (back < 0) back += ring;
  const int q = block + m - back;
  if (q < block) return -1;
  const int first_block = max(1, pos / block - (window - 1));
  return q >= first_block * block ? q : -1;
}

// One CTA per (sample, group of HPC heads); warp w owns cache slots [32w, 32w + 32): one slot per lane for the scores,
// then the warp accumulates its 32 slots' share of p v with coalesced value-row reads and the CTA adds the partial
// sums.
template <typename T, int DH, int HPC>
__global__ void __launch_bounds__(480) decode_attn_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                           const T* __restrict__ v, const float* __restrict__ cos_t,
                                                           const float* __restrict__ sin_t, T* __restrict__ key_cache,
                                                           T* __restrict__ value_cache, T* __restrict__ out,
                                                           const int* __restrict__ pos_ptr, int B, int H, int window,
                                                           int block, int table_rows, int64_t in_stride, float scale) {
  constexpr int kVec = 16 / sizeof(T);              // elements per 16-byte load
  constexpr int kMaxWarps = 15;                     // window <= 14
  constexpr int kPer = DH / 32;                     // output features per lane (1, 2 or 4)
  __shared__ float s_q[HPC][DH];
  __shared__ float s_max[HPC][kMaxWarps], s_sum[HPC][kMaxWarps];
  __shared__ float s_out[HPC][kMaxWarps][DH];
  __shared__ float s_score[HPC][kMaxWarps * 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int groups = H / HPC;
  const int b = blockIdx.x / groups, h0 = (blockIdx.x - b * groups) * HPC;
  const int d_model = H * DH;
  const int pos = *pos_ptr;
  const int C = (window + 1) * block;
  const int slot = pos < block ? pos : block + (pos - block) % (window * block);
  const int trow = min(pos, table_rows - 1);

  // ---- warp 0: rotary on the new q / k rows, append k / v --------------------------------------------------------
  const size_t row = (size_t)b * in_stride + (size_t)h0 * DH;         // q / k / v rows may be slices of one [B, 3D] GEMM
  const size_t out_row = (size_t)b * d_model + (size_t)h0 * DH;
  T* kc = key_cache + ((size_t)b * C) * d_model + (size_t)h0 * DH;
  T* vc = value_cache + ((size_t)b * C) * d_model + (size_t)h0 * DH;
  for (int pr = lane; warp == 0 && pr < DH / 2; pr += 32) {     // rotary pair pr (head 128: two per lane)
#pragma unroll
    for (int hh = 0; hh < HPC; ++hh) {
      const int f = hh * DH + 2 * pr;               // feature offset inside this CTA's head group
      const float c = cos_t[(size_t)trow * (d_model / 2) + (h0 * DH + f) / 2];
      const float s = sin_t[(size_t)trow * (d_model / 2) + (h0 * DH + f) / 2];
      const float qe = to_f32<T>(q[row + f]), qo = to_f32<T>(q[row + f + 1]);
      const float ke = to_f32<T>(k[row + f]), ko = to_f32<T>(k[row + f + 1]);
      const T q0 = from_f32<T>(__fsub_rn(__fmul_rn(qe, c), __fmul_rn(qo, s)));
      const T q1 = from_f32<T>(__fadd_rn(__fmul_rn(qo, c), __fmul_rn(qe, s)));
      const T k0 = from_f32<T>(__fsub_rn(__fmul_rn(ke, c), __fmul_rn(ko, s)));
      const T k1 = from_f32<T>(__fadd_rn(__fmul_rn(ko, c), __fmul_rn(ke, s)));
      s_q[hh][2 * pr] = to_f32<T>(q0);
      s_q[hh][2 * pr + 1] = to_f32<T>(q1);
      kc[(size_t)slot * d_model + f] = k0;
      kc[(size_t)slot * d_model + f + 1] = k1;
      vc[(size_t)slot * d_model + f] = v[row + f];
      vc[(size_t)slot * d_model + f + 1] = v[row + f + 1];
    }
  }
  __syncthreads();                                  // the CTA sees the appended row (global) and the rotated query

  // ---- scores: one cache slot per lane -----------------------------------------------------------------------------
  const int my_slot = warp * 32 + lane;
  const bool live = my_slot < C && slot_position(my_slot, pos, block, window) >= 0;
  const T* kr = kc + (size_t)my_slot * d_model;
#pragma unroll 1                                    // one head's 8 row loads at a time: registers buy CTAs per SM here
  for (int hh = 0; hh < HPC; ++hh) {
    float sc = -INFINITY;
    if (live) {
      DPack<T, kVec> kv[DH / kVec];
#pragma unroll
      for (int i = 0; i < DH / kVec; ++i) kv[i] = *reinterpret_cast<const DPack<T, kVec>*>(kr + hh * DH + i * kVec);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < DH / kVec; ++i)
#pragma unroll
        for (int e = 0; e < kVec; ++e) acc = fmaf(s_q[hh][i * kVec + e], to_f32<T>(kv[i].v[e]), acc);
      sc = acc * scale;
    }
    s_score[hh][threadIdx.x] = sc;
    float wmax = sc;
#pragma unroll
    for (int o = 16; o; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    if (lane == 0) s_max[hh][warp] = wmax;
  }
  __syncthreads();
  float p[HPC];
  bool any = false;
#pragma unroll
  for (int hh = 0; hh < HPC; ++hh) {
    float row_max = -INFINITY;
    for (int w = 0; w < nwarps; ++w) row_max = fmaxf(row_max, s_max[hh][w]);    // the newest key is always live: finite
    const float sc = s_score[hh][threadIdx.x];
    p[hh] = sc == -INFINITY ? 0.f : __expf(sc - row_max);
    float wsum = p[hh];
#pragma unroll
    for (int o = 16; o; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    if (lane == 0) s_sum[hh][warp] = wsum;
    any |= wsum != 0.f;
  }

  // ---- this warp's share of p v: coalesced value rows, lanes split each head's features ---------------------------
  float acc[HPC][kPer] = {};
  if (any) {
    // no per-slot branch: empty / evicted slots hold finite values (the cache starts zeroed) and p == 0 there, and
    // unconditional loads keep 16 value rows per head in flight instead of one
    const T* vr = vc + (size_t)(warp * 32) * d_model + lane * kPer;
#pragma unroll
    for (int hh = 0; hh < HPC; ++hh) {
#pragma unroll
      for (int j0 = 0; j0 < 32; j0 += 16) {
        DPack<T, kPer> vv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
          vv[j] = *reinterpret_cast<const DPack<T, kPer>*>(vr + (size_t)(j0 + j) * d_model + hh * DH);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float pj = __shfl_sync(0xffffffffu, p[hh], j0 + j);
#pragma unroll
          for (int e = 0; e < kPer; ++e) acc[hh][e] = fmaf(pj, to_f32<T>(vv[j].v[e]), acc[hh][e]);
        }
      }
    }
  }
#pragma unroll
  for (int hh = 0; hh < HPC; ++hh)
#pragma unroll
    for (int e = 0; e < kPer; ++e) s_out[hh][warp][lane * kPer + e] = acc[hh][e];
  __syncthreads();
  for (int f = threadIdx.x; f < HPC * DH; f += blockDim.x) {
    const int hh = f / DH, d = f - hh * DH;
    float o = 0.f, z = 0.f;
    for (int w = 0; w < nwarps; ++w) {
      o += s_out[hh][w][d];
      z += s_sum[hh][w];
    }
    out[out_row + f] = from_f32<T>(o / z);
  }
}

template <typename T>
static int launch_decode(const void* q, const void* k, const void* v, const float* c, const float* s, void* kc, void* vc,
                         void* out, const int* pos, int B, int H, int Dh, int window, int block, int table_rows,
                         int64_t in_stride, float scale, cudaStream_t st) {
  const unsigned threads = (unsigned)((window + 1) * 32);
#define SVAE_DEC(DH, HPC)                                                                                               \
  decode_attn_kernel<T, DH, HPC><<<(unsigned)(B * (H / HPC)), threads, 0, st>>>(                                        \
      (const T*)q, (const T*)k, (const T*)v, c, s, (T*)kc, (T*)vc, (T*)out, pos, B, H, window, block, table_rows, in_stride, scale)
  // HPC = 2 (half the CTAs, twice the loads in flight per lane) measured slower on B200: 29 us vs 21 us per launch at
  // 256 samples x 8 heads x 160 slots -- its registers cost more residency than the extra loads buy
  if (Dh == 128) SVAE_DEC(128, 1); else if (Dh == 64) SVAE_DEC(64, 1); else SVAE_DEC(32, 1);
#undef SVAE_DEC
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

}  // namespace svae

using namespace svae;

extern "C" int svae_decode_attn_supported(int32_t head_dim, int32_t window, int32_t block) {
  return (head_dim == 32 || head_dim == 64 || head_dim == 128) && window >= 1 && window <= 14 && block == 32;
}

extern "C" int svae_decode_attn(const void* q, const void* k, const void* v, const float* cos_table,
                                const float* sin_table, void* key_cache, void* value_cache, void* out,
                                const int32_t* position, int32_t B, int32_t H, int32_t head_dim, int32_t window,
                                int32_t block, int32_t table_rows, int64_t in_stride, int32_t dtype, float scale,
                                void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SVAE_REQUIRE(q && k && v && cos_table && sin_table && key_cache && value_cache && out && position, SVAE_ERR_INVALID,
               "svae_decode_attn: null argument");
  SVAE_REQUIRE(svae_decode_attn_supported(head_dim, window, block), SVAE_ERR_UNSUPPORTED,
               "svae_decode_attn: head_dim %d / window %d / block %d not supported (head_dim 32|64|128, window 1..14, block 32)",
               head_dim, window, block);
  SVAE_REQUIRE(B >= 0 && H > 0 && table_rows > 0 && in_stride >= (int64_t)H * head_dim && in_stride % 8 == 0,
               SVAE_ERR_INVALID, "svae_decode_attn: bad sizes");
  const uintptr_t a = reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                      reinterpret_cast<uintptr_t>(key_cache) | reinterpret_cast<uintptr_t>(value_cache) |
                      reinterpret_cast<uintptr_t>(out);
  SVAE_REQUIRE((a & 15) == 0, SVAE_ERR_INVALID, "svae_decode_attn: tensors must be 16-byte aligned");
  if (B == 0) return SVAE_OK;
  ScopedKernelTimer timer("decode_attn", st);
  if (dtype == SVAE_DTYPE_F32)
    return launch_decode<float>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, B, H, head_dim,
                                window, block, table_rows, in_stride, scale, st);
  if (dtype == SVAE_DTYPE_BF16)
    return launch_decode<__nv_bfloat16>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, B, H,
                                        head_dim, window, block, table_rows, in_stride, scale, st);
  if (dtype == SVAE_DTYPE_F16)
    return launch_decode<__half>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, B, H, head_dim,
                                 window, block, table_rows, in_stride, scale, st);
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_decode_attn: dtype %d", dtype);
}
