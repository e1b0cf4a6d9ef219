// Token-by-token decoding step of one DENSE causal attention layer (reference core/attention.py:60-100 with the
// growing KV cache of :107-142, `cfg is None`), driven by TransformerVAE.sample and TransformerLanguageModel.sample.
//
// The counterpart of decode_attn.cu for decoders without block-sparse attention.  The cache is the reference's
// [B, cache_len, d_model] buffer in which slot p holds position p (no ring), so the step reads every slot 0..p:
// 2 * B * (p+1) * d_model * sizeof(T) bytes per launch, growing with the position.  One query row per (sample, head)
// makes it ~2 FLOP per byte: HBM-bound, and what matters is how many independent loads are in flight.
//
// Split-KV.  The live slots 0..p are cut into tiles of kTile slots; the tiles are dealt out in contiguous runs to
// `splits` CTAs per (sample, head) -- a count the host fixes from B, H and cache_len (enough CTAs to fill the GPU) so
// that the grid, and hence a captured graph, does not depend on the position.  Each CTA
//   * rotates the new query row itself (fp32 tables, one rounding to T -- the arithmetic of decode_attn_kernel),
//   * if it owns the tile holding p: rotates the new key row and appends k / v at slot p, then reads them back with
//     the rest of its tiles,
//   * runs an online softmax over its tiles: per tile, half a key row per thread (two threads per slot) and the value
//     rows as 16-byte column vectors (kTile / groups rows per thread), all issued before the first score is reduced,
//   * writes its running max, sum and unnormalised fp32 output to the workspace.
// A second launch merges the partials of each (sample, head) in split order: no atomics, so the result is a function of
// the inputs and the position alone and bit-identical from run to run.  With one split the first kernel normalises
// and writes the output itself and the merge is not launched.
#include <algorithm>

#include "common.cuh"

namespace svae {

namespace {

constexpr int kThreads = 256;
constexpr int kKeySplit = 2;             // threads per key row (two halves of the dot product)
constexpr int kTile = kThreads / kKeySplit;   // slots per tile
constexpr int kMaxCacheLen = 65536;
constexpr int kTargetCtas = 148 * 8;     // at least this many working CTAs when the batch allows it

template <typename T, int N> struct alignas(sizeof(T) * N) DensePack { T v[N]; };

// splits per (sample, head): enough CTAs to fill the SMs, never more than the tiles a full cache holds
int dense_splits(int B, int H, int cache_len) {
  const int tiles = (cache_len + kTile - 1) / kTile;
  const long long pairs = (long long)B * H;
  const long long want = pairs > 0 ? (kTargetCtas + pairs - 1) / pairs : 1;
  return (int)std::max<long long>(1, std::min<long long>(want, tiles));
}

// tiles [first, last) of split s at position pos; empty when the split has nothing to do
__device__ __forceinline__ void split_tiles(int pos, int splits, int s, int& first, int& last, int& per) {
  const int tiles = pos / kTile + 1;
  per = (tiles + splits - 1) / splits;
  first = s * per;
  last = min(first + per, tiles);
}

}  // namespace

// grid (B * H, splits), kThreads threads
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) decode_attn_dense_kernel(
    const T* __restrict__ q, const T* __restrict__ k, const T* __restrict__ v, const float* __restrict__ cos_t,
    const float* __restrict__ sin_t, T* key_cache, T* value_cache, T* __restrict__ out, const int* __restrict__ pos_ptr,
    float* __restrict__ ws_max, float* __restrict__ ws_sum, float* __restrict__ ws_out, int H, int cache_len,
    int table_rows, int64_t in_stride, float scale) {
  constexpr int kVec = 16 / sizeof(T);              // elements per 16-byte load
  constexpr int kCols = DH / kVec;                  // 16-byte vectors per head row
  constexpr int kGroups = kThreads / kCols;         // value rows handled side by side
  constexpr int kRows = kTile / kGroups;            // value rows per thread and tile
  constexpr int kWarps = kThreads / 32;
  __shared__ float s_q[DH];
  __shared__ float s_p[kTile];
  __shared__ float s_red[kWarps];
  __shared__ float s_acc[kGroups][DH + 1];

  const int pos = *pos_ptr;
  if (pos < 0 || pos >= cache_len) return;          // nothing is read or written outside the buffers
  const int splits = gridDim.y, s = blockIdx.y;
  int first, last, per;
  split_tiles(pos, splits, s, first, last, per);
  if (first >= last) return;                        // every slot of this split lies after the position
  const int bh = blockIdx.x, b = bh / H, h = bh - b * H;
  const int d_model = H * DH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int trow = min(pos, table_rows - 1);
  const size_t row = (size_t)b * in_stride + (size_t)h * DH;
  T* kc = key_cache + (size_t)b * cache_len * d_model + (size_t)h * DH;
  T* vc = value_cache + (size_t)b * cache_len * d_model + (size_t)h * DH;
  const bool owner = last * kTile > pos;            // the split holding slot pos appends the new row

  // ---- rotary on the new q (and k) row; the owner appends k / v at slot pos ----------------------------------------
  if (tid < DH / 2) {
    const int f = 2 * tid;
    const float c = cos_t[(size_t)trow * (d_model / 2) + (h * DH + f) / 2];
    const float sn = sin_t[(size_t)trow * (d_model / 2) + (h * DH + f) / 2];
    const float qe = to_f32<T>(q[row + f]), qo = to_f32<T>(q[row + f + 1]);
    s_q[f] = to_f32<T>(from_f32<T>(__fsub_rn(__fmul_rn(qe, c), __fmul_rn(qo, sn))));
    s_q[f + 1] = to_f32<T>(from_f32<T>(__fadd_rn(__fmul_rn(qo, c), __fmul_rn(qe, sn))));
    if (owner) {
      const float ke = to_f32<T>(k[row + f]), ko = to_f32<T>(k[row + f + 1]);
      kc[(size_t)pos * d_model + f] = from_f32<T>(__fsub_rn(__fmul_rn(ke, c), __fmul_rn(ko, sn)));
      kc[(size_t)pos * d_model + f + 1] = from_f32<T>(__fadd_rn(__fmul_rn(ko, c), __fmul_rn(ke, sn)));
      vc[(size_t)pos * d_model + f] = v[row + f];
      vc[(size_t)pos * d_model + f + 1] = v[row + f + 1];
    }
  }
  __syncthreads();                                  // the CTA sees the appended row (global) and the rotated query

  float run_max = -INFINITY, run_sum = 0.f;
  float acc[kVec];
#pragma unroll
  for (int e = 0; e < kVec; ++e) acc[e] = 0.f;
  const int col = tid % kCols, group = tid / kCols;

  for (int tile = first; tile < last; ++tile) {
    const int base = tile * kTile;
    // every load of the tile is issued before any of them is used: half a key row (Dh / kVec / 2 16-byte vectors) and
    // kRows value vectors per thread
    const int my_slot = base + tid / kKeySplit, half = tid % kKeySplit;
    const bool live = my_slot <= pos;
    DensePack<T, kVec> kv[kCols / kKeySplit], vv[kRows];
    const T* kr = kc + (size_t)my_slot * d_model + half * (DH / kKeySplit);
#pragma unroll
    for (int i = 0; i < kCols / kKeySplit; ++i) {
      if (live) kv[i] = *reinterpret_cast<const DensePack<T, kVec>*>(kr + i * kVec);
      else kv[i] = DensePack<T, kVec>{};
    }
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
      const int slot = base + group + j * kGroups;
      if (slot <= pos) vv[j] = *reinterpret_cast<const DensePack<T, kVec>*>(vc + (size_t)slot * d_model + col * kVec);
      else vv[j] = DensePack<T, kVec>{};
    }
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < kCols / kKeySplit; ++i)
#pragma unroll
      for (int e = 0; e < kVec; ++e) dot = fmaf(s_q[half * (DH / kKeySplit) + i * kVec + e], to_f32<T>(kv[i].v[e]), dot);
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);    // both threads of the row hold the same sum
    const float sc = live ? dot * scale : -INFINITY;
    // tile max, in a fixed order
    float m = sc;
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_red[warp] = m;
    __syncthreads();
    float tile_max = -INFINITY;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) tile_max = fmaxf(tile_max, s_red[w]);
    const float new_max = fmaxf(run_max, tile_max);  // finite: slot `base` <= pos is live
    const float alpha = run_max == -INFINITY ? 0.f : __expf(run_max - new_max);
    const float p = live ? __expf(sc - new_max) : 0.f;
    if (half == 0) s_p[tid / kKeySplit] = p;
    float psum = half == 0 ? p : 0.f;
#pragma unroll
    for (int o = 16; o; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
    __syncthreads();                                // s_red (max) read by all, s_p complete
    if (lane == 0) s_red[warp] = psum;
    __syncthreads();
    float tile_sum = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) tile_sum += s_red[w];
    run_sum = run_sum * alpha + tile_sum;
    run_max = new_max;
#pragma unroll
    for (int e = 0; e < kVec; ++e) acc[e] *= alpha;
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
      const float pj = s_p[group + j * kGroups];
#pragma unroll
      for (int e = 0; e < kVec; ++e) acc[e] = fmaf(pj, to_f32<T>(vv[j].v[e]), acc[e]);
    }
    __syncthreads();                                // s_p / s_red are rewritten by the next tile
  }

  // ---- this CTA's output row: the groups' partial sums added in group order ----------------------------------------
#pragma unroll
  for (int e = 0; e < kVec; ++e) s_acc[group][col * kVec + e] = acc[e];
  __syncthreads();
  if (tid < DH) {
    float o = 0.f;
    for (int g = 0; g < kGroups; ++g) o += s_acc[g][tid];
    if (splits == 1) {
      out[(size_t)b * d_model + (size_t)h * DH + tid] = from_f32<T>(o / run_sum);
    } else {
      const size_t slot = (size_t)bh * splits + s;
      ws_out[slot * DH + tid] = o;
      if (tid == 0) {
        ws_max[slot] = run_max;
        ws_sum[slot] = run_sum;
      }
    }
  }
}

// grid B * H, DH threads: out = sum_s exp(m_s - M) o_s / sum_s exp(m_s - M) l_s over the working splits, in split order
template <typename T, int DH>
__global__ void __launch_bounds__(DH) decode_attn_dense_merge_kernel(const float* __restrict__ ws_max,
                                                                      const float* __restrict__ ws_sum,
                                                                      const float* __restrict__ ws_out, T* __restrict__ out,
                                                                      const int* __restrict__ pos_ptr, int H,
                                                                      int cache_len, int splits) {
  const int pos = *pos_ptr;
  if (pos < 0 || pos >= cache_len) return;
  int first, last, per;
  split_tiles(pos, splits, 0, first, last, per);
  const int working = (pos / kTile + 1 + per - 1) / per;
  const int bh = blockIdx.x, d = threadIdx.x;
  const size_t base = (size_t)bh * splits;
  float M = -INFINITY;
  for (int s = 0; s < working; ++s) M = fmaxf(M, ws_max[base + s]);
  float L = 0.f, O = 0.f;
  for (int s = 0; s < working; ++s) {
    const float w = __expf(ws_max[base + s] - M);
    L = fmaf(w, ws_sum[base + s], L);
    O = fmaf(w, ws_out[(base + s) * DH + d], O);
  }
  out[(size_t)bh * DH + d] = from_f32<T>(O / L);
}

template <typename T>
static int launch_decode_dense(const void* q, const void* k, const void* v, const float* c, const float* s, void* kc,
                               void* vc, void* out, const int* pos, float* ws, int B, int H, int Dh, int cache_len,
                               int table_rows, int64_t in_stride, float scale, cudaStream_t st) {
  const int splits = dense_splits(B, H, cache_len);
  const size_t parts = (size_t)B * H * splits;
  float* ws_max = splits > 1 ? ws : nullptr;
  float* ws_sum = splits > 1 ? ws + parts : nullptr;
  float* ws_out = splits > 1 ? ws + 2 * parts : nullptr;
  const dim3 grid((unsigned)(B * H), (unsigned)splits);
#define SVAE_DEC_DENSE(DH)                                                                                               \
  do {                                                                                                                   \
    decode_attn_dense_kernel<T, DH><<<grid, kThreads, 0, st>>>((const T*)q, (const T*)k, (const T*)v, c, s, (T*)kc,      \
                                                               (T*)vc, (T*)out, pos, ws_max, ws_sum, ws_out, H,          \
                                                               cache_len, table_rows, in_stride, scale);                 \
    if (splits > 1)                                                                                                      \
      decode_attn_dense_merge_kernel<T, DH><<<(unsigned)(B * H), DH, 0, st>>>(ws_max, ws_sum, ws_out, (T*)out, pos, H,   \
                                                                              cache_len, splits);                        \
  } while (0)
  if (Dh == 64) SVAE_DEC_DENSE(64); else SVAE_DEC_DENSE(32);
#undef SVAE_DEC_DENSE
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

}  // namespace svae

using namespace svae;

extern "C" int svae_decode_attn_dense_supported(int32_t head_dim, int32_t cache_len) {
  return (head_dim == 32 || head_dim == 64) && cache_len >= 1 && cache_len <= kMaxCacheLen;
}

extern "C" size_t svae_decode_attn_dense_workspace_bytes(int32_t B, int32_t H, int32_t head_dim, int32_t cache_len) {
  if (B <= 0 || H <= 0 || !svae_decode_attn_dense_supported(head_dim, cache_len)) return 0;
  const int splits = dense_splits(B, H, cache_len);
  return splits > 1 ? (size_t)B * H * splits * (head_dim + 2) * sizeof(float) : 0;
}

extern "C" int svae_decode_attn_dense(const void* q, const void* k, const void* v, const float* cos_table,
                                      const float* sin_table, void* key_cache, void* value_cache, void* out,
                                      const int32_t* position, void* workspace, size_t workspace_bytes, int32_t B,
                                      int32_t H, int32_t head_dim, int32_t cache_len, int32_t table_rows,
                                      int64_t in_stride, int32_t dtype, float scale, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SVAE_REQUIRE(q && k && v && cos_table && sin_table && key_cache && value_cache && out && position, SVAE_ERR_INVALID,
               "svae_decode_attn_dense: null argument");
  SVAE_REQUIRE(svae_decode_attn_dense_supported(head_dim, cache_len), SVAE_ERR_UNSUPPORTED,
               "svae_decode_attn_dense: head_dim %d / cache_len %d not supported (head_dim 32|64, cache_len 1..%d)",
               head_dim, cache_len, kMaxCacheLen);
  SVAE_REQUIRE(B >= 0 && H > 0 && (int64_t)B * H <= INT32_MAX && table_rows > 0 &&
                   in_stride >= (int64_t)H * head_dim && in_stride % 8 == 0,
               SVAE_ERR_INVALID, "svae_decode_attn_dense: bad sizes");
  const size_t need = svae_decode_attn_dense_workspace_bytes(B, H, head_dim, cache_len);
  SVAE_REQUIRE(workspace_bytes >= need && (need == 0 || workspace), SVAE_ERR_INVALID,
               "svae_decode_attn_dense: workspace of %zu bytes, %zu needed", workspace_bytes, need);
  const uintptr_t a = reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                      reinterpret_cast<uintptr_t>(key_cache) | reinterpret_cast<uintptr_t>(value_cache) |
                      reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(workspace);
  SVAE_REQUIRE((a & 15) == 0, SVAE_ERR_INVALID, "svae_decode_attn_dense: tensors must be 16-byte aligned");
  if (B == 0) return SVAE_OK;
  ScopedKernelTimer timer("decode_attn_dense", st);
  float* ws = reinterpret_cast<float*>(workspace);
  if (dtype == SVAE_DTYPE_F32)
    return launch_decode_dense<float>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, ws, B, H,
                                      head_dim, cache_len, table_rows, in_stride, scale, st);
  if (dtype == SVAE_DTYPE_BF16)
    return launch_decode_dense<__nv_bfloat16>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, ws,
                                              B, H, head_dim, cache_len, table_rows, in_stride, scale, st);
  if (dtype == SVAE_DTYPE_F16)
    return launch_decode_dense<__half>(q, k, v, cos_table, sin_table, key_cache, value_cache, out, position, ws, B, H,
                                       head_dim, cache_len, table_rows, in_stride, scale, st);
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_decode_attn_dense: dtype %d", dtype);
}
