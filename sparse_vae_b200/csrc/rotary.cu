// Rotary position encoding of the q / k projections feeding the sparse-attention kernel, one launch per tensor
// (SURVEY.md section 8f row 1; reference core/attention.py:194-208 `encode_position_rotary`, called at :61,70).
//
// The reference rotates consecutive feature pairs over the FULL d_model before the head split, and evaluates
// everything in the activation dtype (positions, angles, cos/sin and every product / sum are rounded to bf16 under
// autocast).  The host side builds the [L, d/2] cos / sin tables with exactly those torch ops; this kernel then
// applies
//     out[2i]   = rn(rn(x[2i] * cos_i) - rn(x[2i+1] * sin_i))
//     out[2i+1] = rn(rn(x[2i+1] * cos_i) + rn(x[2i] * sin_i))
// with one rounding per product and per sum, i.e. bit-identical to the reference's ~10 element-wise launches on
// strided views.  `conj = 1` rotates by the negative angle, which is exactly autograd's backward of the above
// (d even = rn(rn(g_e c) + rn(g_o s)), d odd = rn(rn(g_o c) - rn(g_e s))).
// HBM-bound: 2 * rows * d * sizeof(T) bytes per launch (tables stay in L2).
#include <type_traits>

#include "common.cuh"

namespace svae {

template <typename T> struct RotOps;
template <> struct RotOps<float> {
  using V = float;
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }   // no FMA contraction
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
};
template <> struct RotOps<__nv_bfloat16> {
  static __device__ __forceinline__ __nv_bfloat16 mul(__nv_bfloat16 a, __nv_bfloat16 b) {
    return __float2bfloat16_rn(__bfloat162float(a) * __bfloat162float(b));                    // exact product, one rounding
  }
  static __device__ __forceinline__ __nv_bfloat16 add(__nv_bfloat16 a, __nv_bfloat16 b) {
    return __float2bfloat16_rn(__bfloat162float(a) + __bfloat162float(b));
  }
  static __device__ __forceinline__ __nv_bfloat16 sub(__nv_bfloat16 a, __nv_bfloat16 b) {
    return __float2bfloat16_rn(__bfloat162float(a) - __bfloat162float(b));
  }
};
template <> struct RotOps<__half> {
  static __device__ __forceinline__ __half mul(__half a, __half b) { return __float2half_rn(__half2float(a) * __half2float(b)); }
  static __device__ __forceinline__ __half add(__half a, __half b) { return __float2half_rn(__half2float(a) + __half2float(b)); }
  static __device__ __forceinline__ __half sub(__half a, __half b) { return __float2half_rn(__half2float(a) - __half2float(b)); }
};

template <typename T, int N> struct alignas(sizeof(T) * N) Pack { T v[N]; };

template <typename T> __device__ __forceinline__ float rot_to_f32(T v);
template <> __device__ __forceinline__ float rot_to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float rot_to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float rot_to_f32<float>(float v) { return v; }

template <typename T, typename TT>
__device__ __forceinline__ Pack<T, 8> rotate8(const Pack<T, 8>& xv, const Pack<TT, 4>& c, const Pack<TT, 4>& s, int conj);

// one thread = 8 consecutive features (4 pairs) of one row.
// TT == T : every op rounded to T (the reference outside autocast).
// TT == float, T 16-bit : the reference UNDER AUTOCAST -- `pow` is an fp32 autocast op, so cos / sin are fp32 and the
//   products promote to fp32: forward = fp32 products and difference, rounded to T once (the rounding the consuming
//   matmul's autocast cast applies); backward = autograd of the promoted products: each fp32 product is cast back
//   to T and the two contributions are summed in T.
template <typename T, typename TT>
__global__ void __launch_bounds__(256) rotary_kernel(const T* x, const TT* __restrict__ cos_t,      // (x may alias out)
                                                      const TT* __restrict__ sin_t, T* out, int64_t rows, int L,
                                                      int d, int conj, int64_t in_ld, int64_t out_ld) {
  const int vec_per_row = d >> 3;
  const int64_t total = rows * vec_per_row;
  const int half = d >> 1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / vec_per_row;
    const int vcol = (int)(i - r * vec_per_row);
    const int pos = (int)(r % L);
    const Pack<T, 8> xv = *reinterpret_cast<const Pack<T, 8>*>(x + r * in_ld + vcol * 8);
    const Pack<TT, 4> c = *reinterpret_cast<const Pack<TT, 4>*>(cos_t + (int64_t)pos * half + vcol * 4);
    const Pack<TT, 4> s = *reinterpret_cast<const Pack<TT, 4>*>(sin_t + (int64_t)pos * half + vcol * 4);
    *reinterpret_cast<Pack<T, 8>*>(out + r * out_ld + vcol * 8) = rotate8<T, TT>(xv, c, s, conj);
  }
}

template <typename T, typename TT>
__device__ __forceinline__ Pack<T, 8> rotate8(const Pack<T, 8>& xv, const Pack<TT, 4>& c, const Pack<TT, 4>& s, int conj) {
  constexpr bool kMixed = !std::is_same<T, TT>::value;
  Pack<T, 8> o;
  {
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      if constexpr (!kMixed) {
        const T e = xv.v[2 * p], od = xv.v[2 * p + 1];
        const T ec = RotOps<T>::mul(e, c.v[p]), os = RotOps<T>::mul(od, s.v[p]);
        const T oc = RotOps<T>::mul(od, c.v[p]), es = RotOps<T>::mul(e, s.v[p]);
        if (!conj) {
          o.v[2 * p] = RotOps<T>::sub(ec, os);
          o.v[2 * p + 1] = RotOps<T>::add(oc, es);
        } else {
          o.v[2 * p] = RotOps<T>::add(ec, os);
          o.v[2 * p + 1] = RotOps<T>::sub(oc, es);
        }
      } else {
        const float e = rot_to_f32<T>(xv.v[2 * p]), od = rot_to_f32<T>(xv.v[2 * p + 1]);
        const float cf = c.v[p], sf = s.v[p];
        const float ec = __fmul_rn(e, cf), os = __fmul_rn(od, sf), oc = __fmul_rn(od, cf), es = __fmul_rn(e, sf);
        if (!conj) {
          o.v[2 * p] = from_f32<T>(__fsub_rn(ec, os));
          o.v[2 * p + 1] = from_f32<T>(__fadd_rn(oc, es));
        } else {
          o.v[2 * p] = RotOps<T>::add(from_f32<T>(ec), from_f32<T>(os));
          o.v[2 * p + 1] = RotOps<T>::sub(from_f32<T>(oc), from_f32<T>(es));
        }
      }
    }
  }
  return o;
}

// ---- q and k of one attention layer in ONE launch, optionally with the column sums of both outputs ---------------
// (the bias gradients of the q / k projections when the launch is the backward rotation of dq / dk: core/linear.py
// `qkv_rotary`).  Work layout, accumulation order and final reduction are those of colsum_partial_kernel
// (csrc/colsum.cu), so the sums are bit-identical to `svae_colsum` of the rotated tensors; the rotation itself is
// rotate8 above, bit-identical to two `svae_rotary` launches.
template <typename T, typename TT, bool kSums>
__global__ void __launch_bounds__(256) rotary_pair_kernel(const T* xa, const T* xb,      // (may alias oa / ob: no __restrict__)
                                                           const TT* __restrict__ cos_t, const TT* __restrict__ sin_t,
                                                           T* oa, T* ob, int64_t rows, int L, int d, int conj, int64_t in_ld,
                                                           int64_t out_ld,
                                                           float* __restrict__ partial, unsigned* __restrict__ counters,
                                                           float* __restrict__ sum_a, float* __restrict__ sum_b) {
  __shared__ float red[kSums ? 8 : 1][32][17];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int vec = blockIdx.x * 32 + cx;
  const bool ok = vec * 8 < d;
  const int half = d >> 1;
  float acc[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) acc[e] = 0.f;
  auto one = [&](int64_t r, const Pack<T, 8>& va, const Pack<T, 8>& vb) {
    const int pos = (int)(r % L);
    const int64_t off = r * out_ld + vec * 8;
    const Pack<TT, 4> c = *reinterpret_cast<const Pack<TT, 4>*>(cos_t + (int64_t)pos * half + vec * 4);
    const Pack<TT, 4> s = *reinterpret_cast<const Pack<TT, 4>*>(sin_t + (int64_t)pos * half + vec * 4);
    const Pack<T, 8> ra = rotate8<T, TT>(va, c, s, conj), rb = rotate8<T, TT>(vb, c, s, conj);
    *reinterpret_cast<Pack<T, 8>*>(oa + off) = ra;
    *reinterpret_cast<Pack<T, 8>*>(ob + off) = rb;
    if constexpr (kSums) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        acc[e] += rot_to_f32<T>(ra.v[e]);
        acc[8 + e] += rot_to_f32<T>(rb.v[e]);
      }
    }
  };
  if (ok) {
    // software pipeline: the tensor loads of the next pair of rows are in flight while this pair is rotated (the rows are
    // visited, and their values accumulated, in the order of colsum_partial_kernel: r, r + step, r + 2 step, ...)
    const int64_t step = (int64_t)gridDim.y * 8;
    int64_t r = (int64_t)blockIdx.y * 8 + ry;
    auto ld = [&](const T* p, int64_t row) {
      Pack<T, 8> v;
      if (row < rows) v = *reinterpret_cast<const Pack<T, 8>*>(p + row * in_ld + vec * 8);
      return v;
    };
    Pack<T, 8> a0 = ld(xa, r), b0 = ld(xb, r), a1 = ld(xa, r + step), b1 = ld(xb, r + step);
    for (; r < rows; r += 2 * step) {
      const int64_t rn = r + 2 * step;
      const Pack<T, 8> na0 = ld(xa, rn), nb0 = ld(xb, rn), na1 = ld(xa, rn + step), nb1 = ld(xb, rn + step);
      one(r, a0, b0);
      if (r + step < rows) one(r + step, a1, b1);
      a0 = na0; b0 = nb0; a1 = na1; b1 = nb1;
    }
  }
  if constexpr (kSums) {
    const int64_t plane = (int64_t)gridDim.y * d;            // partial: [2][slabs][d]
#pragma unroll
    for (int e = 0; e < 16; ++e) red[ry][cx][e] = acc[e];
    __syncthreads();
    if (ry == 0 && ok) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][cx][e];
        partial[(e >> 3) * plane + (int64_t)blockIdx.y * d + vec * 8 + (e & 7)] = t;
      }
    }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&counters[blockIdx.x], 1u) == gridDim.y - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
#pragma unroll
    for (int e = 0; e < 16; ++e) acc[e] = 0.f;
    if (ok)
      for (int b = ry; b < (int)gridDim.y; b += 8) {
#pragma unroll
        for (int t2 = 0; t2 < 2; ++t2) {
          const float* src = partial + t2 * plane + (int64_t)b * d + vec * 8;
          const float4 u = __ldcg(reinterpret_cast<const float4*>(src)), w = __ldcg(reinterpret_cast<const float4*>(src + 4));
          acc[8 * t2 + 0] += u.x; acc[8 * t2 + 1] += u.y; acc[8 * t2 + 2] += u.z; acc[8 * t2 + 3] += u.w;
          acc[8 * t2 + 4] += w.x; acc[8 * t2 + 5] += w.y; acc[8 * t2 + 6] += w.z; acc[8 * t2 + 7] += w.w;
        }
      }
#pragma unroll
    for (int e = 0; e < 16; ++e) red[ry][cx][e] = acc[e];
    __syncthreads();
    if (ry == 0 && ok) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][cx][e];
        (e < 8 ? sum_a : sum_b)[vec * 8 + (e & 7)] = t;
      }
    }
    if (threadIdx.x == 0) counters[blockIdx.x] = 0u;
  }
}

// slab count of svae_colsum (csrc/colsum.cu `colsum_slabs`): the same partition of the rows gives the same sums
static int rotary_pair_slabs(int64_t rows, int n) {
  const int col_blocks = (n / 8 + 31) / 32;
  int slabs = (148 * 4 + col_blocks - 1) / col_blocks;
  const int64_t max_slabs = (rows + 63) / 64;
  if (slabs > max_slabs) slabs = (int)(max_slabs > 0 ? max_slabs : 1);
  return slabs;
}

template <typename T, typename TT>
static int launch_rotary_pair(const void* xa, const void* xb, const void* c, const void* s, void* oa, void* ob, int64_t rows, int L,
                              int d, int conj, int64_t in_ld, int64_t out_ld, float* partial, unsigned* counters, float* sum_a,
                              float* sum_b, cudaStream_t st) {
  dim3 grid((d / 8 + 31) / 32, rotary_pair_slabs(rows, d));
  if (sum_a)
    rotary_pair_kernel<T, TT, true><<<grid, 256, 0, st>>>((const T*)xa, (const T*)xb, (const TT*)c, (const TT*)s, (T*)oa, (T*)ob, rows, L, d,
                                                          conj, in_ld, out_ld, partial, counters, sum_a, sum_b);
  else
    rotary_pair_kernel<T, TT, false><<<grid, 256, 0, st>>>((const T*)xa, (const T*)xb, (const TT*)c, (const TT*)s, (T*)oa, (T*)ob, rows, L,
                                                           d, conj, in_ld, out_ld, nullptr, nullptr, nullptr, nullptr);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

template <typename T, typename TT>
static int launch_rotary(const void* x, const void* c, const void* s, void* out, int64_t rows, int L, int d, int conj,
                         int64_t in_ld, int64_t out_ld, cudaStream_t st) {
  const int64_t total = rows * (d >> 3);
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  rotary_kernel<T, TT><<<(unsigned)blocks, 256, 0, st>>>((const T*)x, (const TT*)c, (const TT*)s, (T*)out, rows, L, d, conj, in_ld, out_ld);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

}  // namespace svae

using namespace svae;

static int rotary_ld(const void* x, const void* cos_table, const void* sin_table, void* out, int32_t dtype, int32_t table_dtype,
                     int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj, int64_t in_ld, int64_t out_ld, void* stream);

extern "C" int svae_rotary(const void* x, const void* cos_table, const void* sin_table, void* out, int32_t dtype,
                           int32_t table_dtype, int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj, void* stream) {
  return rotary_ld(x, cos_table, sin_table, out, dtype, table_dtype, rows, seq_len, d_model, conj, d_model, d_model, stream);
}

static int rotary_ld(const void* x, const void* cos_table, const void* sin_table, void* out, int32_t dtype, int32_t table_dtype,
                     int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj, int64_t in_ld, int64_t out_ld, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SVAE_REQUIRE(in_ld >= d_model && out_ld >= d_model && in_ld % 8 == 0 && out_ld % 8 == 0, SVAE_ERR_INVALID,
               "svae_rotary: row strides must be >= d_model and multiples of 8");
  SVAE_REQUIRE(x && cos_table && sin_table && out && rows >= 0, SVAE_ERR_INVALID, "svae_rotary: null argument");
  SVAE_REQUIRE(d_model > 0 && d_model % 8 == 0 && seq_len > 0 && rows % seq_len == 0, SVAE_ERR_INVALID,
               "svae_rotary: d_model must be a multiple of 8 and rows a multiple of seq_len");
  SVAE_REQUIRE(table_dtype == dtype || table_dtype == SVAE_DTYPE_F32, SVAE_ERR_INVALID,
               "svae_rotary: tables must have the tensor's dtype or be fp32 (autocast), got %d / %d", dtype, table_dtype);
  const uintptr_t xa = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out);
  const uintptr_t ta = reinterpret_cast<uintptr_t>(cos_table) | reinterpret_cast<uintptr_t>(sin_table);
  SVAE_REQUIRE((xa & (dtype == SVAE_DTYPE_F32 ? 31 : 15)) == 0 && (ta & (table_dtype == SVAE_DTYPE_F32 ? 15 : 7)) == 0,
               SVAE_ERR_INVALID, "svae_rotary: misaligned tensor");
  if (rows == 0) return SVAE_OK;
  ScopedKernelTimer timer("rotary", st);
#define SVAE_ROT(T, TT) return launch_rotary<T, TT>(x, cos_table, sin_table, out, rows, seq_len, d_model, conj, in_ld, out_ld, st)
  if (dtype == SVAE_DTYPE_F32) SVAE_ROT(float, float);
  if (dtype == SVAE_DTYPE_BF16) { if (table_dtype == dtype) SVAE_ROT(__nv_bfloat16, __nv_bfloat16); SVAE_ROT(__nv_bfloat16, float); }
  if (dtype == SVAE_DTYPE_F16) { if (table_dtype == dtype) SVAE_ROT(__half, __half); SVAE_ROT(__half, float); }
#undef SVAE_ROT
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_rotary: dtype %d", dtype);
}

extern "C" int64_t svae_rotary_pair_workspace_floats(int64_t rows, int32_t d_model) {
  return 2 * (int64_t)rotary_pair_slabs(rows, d_model) * d_model;
}

extern "C" int svae_rotary_pair(const void* xa, const void* xb, const void* cos_table, const void* sin_table, void* oa, void* ob,
                                int32_t dtype, int32_t table_dtype, int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj,
                                int64_t in_ld, int64_t out_ld, float* sum_a, float* sum_b, float* workspace, int64_t workspace_floats,
                                uint32_t* counters, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SVAE_REQUIRE(in_ld >= d_model && out_ld >= d_model && in_ld % 8 == 0 && out_ld % 8 == 0, SVAE_ERR_INVALID,
               "svae_rotary_pair: row strides must be >= d_model and multiples of 8");
  SVAE_REQUIRE(xa && xb && cos_table && sin_table && oa && ob && rows >= 0, SVAE_ERR_INVALID, "svae_rotary_pair: null argument");
  SVAE_REQUIRE(d_model > 0 && d_model % 8 == 0 && seq_len > 0 && rows % seq_len == 0, SVAE_ERR_INVALID,
               "svae_rotary_pair: d_model must be a multiple of 8 and rows a multiple of seq_len");
  SVAE_REQUIRE(table_dtype == dtype || table_dtype == SVAE_DTYPE_F32, SVAE_ERR_INVALID,
               "svae_rotary_pair: tables must have the tensors' dtype or be fp32 (autocast), got %d / %d", dtype, table_dtype);
  const uintptr_t xs = reinterpret_cast<uintptr_t>(xa) | reinterpret_cast<uintptr_t>(xb) | reinterpret_cast<uintptr_t>(oa) |
                       reinterpret_cast<uintptr_t>(ob);
  const uintptr_t ta = reinterpret_cast<uintptr_t>(cos_table) | reinterpret_cast<uintptr_t>(sin_table);
  SVAE_REQUIRE((xs & (dtype == SVAE_DTYPE_F32 ? 31 : 15)) == 0 && (ta & (table_dtype == SVAE_DTYPE_F32 ? 15 : 7)) == 0,
               SVAE_ERR_INVALID, "svae_rotary_pair: misaligned tensor");
  SVAE_REQUIRE((sum_a == nullptr) == (sum_b == nullptr), SVAE_ERR_INVALID, "svae_rotary_pair: both column sums or none");
  if (sum_a)
    SVAE_REQUIRE(workspace && counters && workspace_floats >= svae_rotary_pair_workspace_floats(rows, d_model), SVAE_ERR_INVALID,
                 "svae_rotary_pair: column sums need svae_rotary_pair_workspace_floats() floats and zeroed counters");
  if (rows == 0) return SVAE_OK;
  if (!sum_a) {      // no column sums: the flat one-tensor kernel twice (57.6 us against 61.6 us for the slab layout at [65536, 512])
    const int rc = rotary_ld(xa, cos_table, sin_table, oa, dtype, table_dtype, rows, seq_len, d_model, conj, in_ld, out_ld, stream);
    return rc ? rc : rotary_ld(xb, cos_table, sin_table, ob, dtype, table_dtype, rows, seq_len, d_model, conj, in_ld, out_ld, stream);
  }
  ScopedKernelTimer timer("rotary", st);
#define SVAE_ROTP(T, TT) \
  return launch_rotary_pair<T, TT>(xa, xb, cos_table, sin_table, oa, ob, rows, seq_len, d_model, conj, in_ld, out_ld, workspace, counters, \
                                   sum_a, sum_b, st)
  if (dtype == SVAE_DTYPE_F32) SVAE_ROTP(float, float);
  if (dtype == SVAE_DTYPE_BF16) { if (table_dtype == dtype) SVAE_ROTP(__nv_bfloat16, __nv_bfloat16); SVAE_ROTP(__nv_bfloat16, float); }
  if (dtype == SVAE_DTYPE_F16) { if (table_dtype == dtype) SVAE_ROTP(__half, __half); SVAE_ROTP(__half, float); }
#undef SVAE_ROTP
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_rotary_pair: dtype %d", dtype);
}
