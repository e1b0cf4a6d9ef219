// Fused latent bottleneck: (mu | logvar) -> sigma, z = mu + eps*sigma, elementwise KL, per-row KL sum and the
// batch-mean KL, in one launch; and its analytic backward with eps regenerated from Philox (zero bytes).
//
// Reference semantics (paths relative to the reference repo):
//   core/conditional_gaussian.py:19-27   var = exp(logvar); scale = sqrt(var); kl = 0.5*(mu^2 + var - logvar - 1)
//   core/continuous_autoencoder.py:43-47 z = rsample(); raw_kl = kl.flatten(1).sum(-1); kl = (raw_kl/token_counts).mean()
//   torch Normal.rsample                 eps = empty(shape, dtype=loc.dtype).normal_(); z = loc + eps*scale
// The eps stream reproduces ATen's CUDA normal_ (ATen/native/cuda/DistributionTemplates.h:50-92): element li of
// the flattened tensor is drawn by "thread" li mod T (T = 256*grid) as component (li div T) mod 4 of its
// ((li div T) div 4)-th curand_normal4, with curand_init(seed, thread, offset).  curand's own device functions
// (Philox4x32-10 and the __sincosf Box-Muller) are called directly so the bits match torch's.
//
// HBM-bound, element-wise + row reduction: no tensor cores.  One warp owns a latent row (coalesced 128 B
// accesses, warp-shuffle row sum); when T is a multiple of `latent` the four rows that share one Philox
// output (li, li+T, li+2T, li+3T) are processed together so each Philox/Box-Muller evaluation is used 4x,
// which keeps the kernel under the HBM roofline instead of ALU-bound for large inputs.
#include <curand_kernel.h>
#include <curand_philox4x32_x.h>

#include "common.cuh"

namespace svae {

constexpr int kBnThreads = 256;
constexpr int kBnMaxBlocks = 2048;
// workspace layout (floats): [0] = arrival counter (as uint32), [64 .. 64+kBnMaxBlocks) = per-block partials
constexpr int kBnPartialOffset = 64;

struct PhiloxPlan {
  uint64_t seed, offset;
  int64_t T;   // threads of the emulated ATen launch = 256 * grid
  const uint64_t* dev;   // non-null (CUDA-graph replay): seed = dev[0], offset = dev[1] + offset, read on the device
};

__device__ __forceinline__ PhiloxPlan resolve(PhiloxPlan pp) {
  if (pp.dev) { pp.seed = pp.dev[0]; pp.offset += pp.dev[1]; }
  return pp;
}

__host__ inline int64_t aten_grid(int64_t numel, int sm_count, int max_threads_per_sm) {
  int64_t grid = (numel + 255) / 256;
  int64_t cap = (int64_t)sm_count * (max_threads_per_sm / 256);
  return grid < cap ? grid : cap;
}

// One Philox4x32-10 evaluation -> the four normals curand_normal4 would return for (thread, call).
__device__ __forceinline__ float4 normal4_at(const PhiloxPlan& pp, int64_t thread, int64_t call) {
  uint64_t c = pp.offset / 4 + (uint64_t)call;       // offset is a multiple of 4 (checked on the host)
  uint4 ctr = make_uint4((unsigned)c, (unsigned)(c >> 32), (unsigned)thread, (unsigned)((uint64_t)thread >> 32));
  uint2 key = make_uint2((unsigned)pp.seed, (unsigned)(pp.seed >> 32));
  uint4 r = curand_Philox4x32_10(ctr, key);
  float2 a = _curand_box_muller(r.x, r.y);
  float2 b = _curand_box_muller(r.z, r.w);
  return make_float4(a.x, a.y, b.x, b.y);
}

template <typename T> __device__ __forceinline__ float round_through(float x) { return to_f32<T>(from_f32<T>(x)); }

struct BnFwdArgs {
  const void* mulogvar;
  int64_t ld;
  const int64_t* token_counts;
  int64_t rows;
  int latent;
  PhiloxPlan pp;
  float *z, *sigma, *kl_elem, *raw_kl, *kl;
  float* workspace;
  int64_t quads;       // number of warp work items
  int64_t rows_per_T;  // T / latent when SHARE
};

struct BnBwdArgs {
  const void* mulogvar;
  int64_t ld;
  const int64_t* token_counts;
  int64_t rows;
  int latent;
  PhiloxPlan pp;
  const float *dz, *dsigma, *dkl_elem, *draw_kl, *dkl;
  void* dout;
  int64_t ld_out;
  int64_t quads;
  int64_t rows_per_T;
};

// Maps work item q -> base row and number of companion rows (1 when !SHARE).
template <bool SHARE>
__device__ __forceinline__ void quad_rows(int64_t q, int64_t rows, int64_t R, int64_t& r0, int& nrow) {
  if (SHARE) {
    int64_t m = q / R, i = q - m * R;
    r0 = 4 * m * R + i;
    nrow = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) nrow += (r0 + j * R < rows) ? 1 : 0;
  } else {
    r0 = q;
    nrow = 1;
  }
}

template <typename T, bool SHARE>
__global__ void __launch_bounds__(kBnThreads) bottleneck_fwd_kernel(BnFwdArgs a) {
  a.pp = resolve(a.pp);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_per_block = kBnThreads / 32;
  const T* __restrict__ in = reinterpret_cast<const T*>(a.mulogvar);
  const int D = a.latent;
  float block_part = 0.f;   // sum over this warp's rows of raw_kl/token_count (lane 0 only)

  for (int64_t q = (int64_t)blockIdx.x * warps_per_block + warp; q < a.quads; q += (int64_t)gridDim.x * warps_per_block) {
    int64_t r0;
    int nrow;
    quad_rows<SHARE>(q, a.rows, a.rows_per_T, r0, nrow);
    float rowsum[4] = {0.f, 0.f, 0.f, 0.f};
    for (int d = lane; d < D; d += 32) {
      float4 n4;
      float nv[4];
      if (SHARE) {
        // r0 = 4*m*R + i  =>  flat index r0*D + d = (4m)*T + (i*D + d) with i*D + d < T: "thread" i*D + d, call m, and the
        // four rows r0 + j*R are its components j = 0..3 -- no division per element
        const int64_t m = r0 / (4 * a.rows_per_T), i = r0 - m * 4 * a.rows_per_T;
        n4 = normal4_at(a.pp, i * D + d, m);
        nv[0] = n4.x; nv[1] = n4.y; nv[2] = n4.z; nv[3] = n4.w;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j < nrow) {
          int64_t row = SHARE ? r0 + j * a.rows_per_T : r0;
          float e;
          if (SHARE) {
            e = nv[j];
          } else {
            int64_t li = row * D + d;
            int64_t k = li / a.pp.T;
            n4 = normal4_at(a.pp, li - k * a.pp.T, k >> 2);
            int comp = (int)(k & 3);
            e = comp == 0 ? n4.x : comp == 1 ? n4.y : comp == 2 ? n4.z : n4.w;
          }
          e = round_through<T>(e);                      // eps is materialised in loc.dtype by normal_()
          float mu = to_f32<T>(in[row * a.ld + d]);
          float lv = to_f32<T>(in[row * a.ld + D + d]);
          float var = expf(lv);
          float sg = sqrtf(var);
          // separate roundings (no FMA) so z and kl match the op-by-op torch evaluation bit for bit
          float zz = __fadd_rn(mu, __fmul_rn(e, sg));
          float kk = __fmul_rn(0.5f, __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(mu, mu), var), lv), -1.0f));
          int64_t o = row * D + d;
          a.z[o] = zz;
          a.sigma[o] = sg;
          if (a.kl_elem) a.kl_elem[o] = kk;
          rowsum[j] += kk;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j < nrow) {
        float s = rowsum[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
          int64_t row = SHARE ? r0 + j * a.rows_per_T : r0;
          a.raw_kl[row] = s;
          block_part += s / (float)a.token_counts[row];
        }
      }
    }
  }

  // deterministic two-level reduction of kl = mean_b(raw_kl[b] / token_counts[b])
  __shared__ float warp_part[kBnThreads / 32];
  __shared__ bool is_last;
  if (lane == 0) warp_part[warp] = block_part;
  __syncthreads();
  unsigned* counter = reinterpret_cast<unsigned*>(a.workspace);
  float* partials = a.workspace + kBnPartialOffset;
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < warps_per_block; ++w) s += warp_part[w];
    partials[blockIdx.x] = s;
    __threadfence();
    unsigned prev = atomicAdd(counter, 1u);
    is_last = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && warp == 0) {
    __threadfence();
    float s = 0.f;
    for (int i = lane; i < (int)gridDim.x; i += 32) s += __ldcg(partials + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      a.kl[0] = s / (float)a.rows;
      *counter = 0u;   // self-cleaning for the next launch
    }
  }
}

template <typename T, bool SHARE>
__global__ void __launch_bounds__(kBnThreads) bottleneck_bwd_kernel(BnBwdArgs a) {
  a.pp = resolve(a.pp);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_per_block = kBnThreads / 32;
  const T* __restrict__ in = reinterpret_cast<const T*>(a.mulogvar);
  T* __restrict__ out = reinterpret_cast<T*>(a.dout);
  const int D = a.latent;
  const float dkl = a.dkl ? a.dkl[0] : 0.f;

  for (int64_t q = (int64_t)blockIdx.x * warps_per_block + warp; q < a.quads; q += (int64_t)gridDim.x * warps_per_block) {
    int64_t r0;
    int nrow;
    quad_rows<SHARE>(q, a.rows, a.rows_per_T, r0, nrow);
    for (int d = lane; d < D; d += 32) {
      float4 n4;
      float nv[4];
      if (SHARE) {
        const int64_t m = r0 / (4 * a.rows_per_T), i = r0 - m * 4 * a.rows_per_T;
        n4 = normal4_at(a.pp, i * D + d, m);
        nv[0] = n4.x; nv[1] = n4.y; nv[2] = n4.z; nv[3] = n4.w;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j < nrow) {
          int64_t row = SHARE ? r0 + j * a.rows_per_T : r0;
          float e;
          if (SHARE) {
            e = nv[j];
          } else {
            int64_t li = row * D + d;
            int64_t k = li / a.pp.T;
            n4 = normal4_at(a.pp, li - k * a.pp.T, k >> 2);
            int comp = (int)(k & 3);
            e = comp == 0 ? n4.x : comp == 1 ? n4.y : comp == 2 ? n4.z : n4.w;
          }
          e = round_through<T>(e);
          float mu = to_f32<T>(in[row * a.ld + d]);
          float lv = to_f32<T>(in[row * a.ld + D + d]);
          float var = expf(lv);
          float sg = sqrtf(var);
          int64_t o = row * D + d;
          float g = dkl / ((float)a.rows * (float)a.token_counts[row]);
          if (a.draw_kl) g += a.draw_kl[row];
          if (a.dkl_elem) g += a.dkl_elem[o];
          float gz = a.dz ? a.dz[o] : 0.f;
          float gs = a.dsigma ? a.dsigma[o] : 0.f;
          float dmu = gz + g * mu;
          float dlv = (gz * e + gs) * 0.5f * sg + g * 0.5f * (var - 1.0f);
          out[row * a.ld_out + d] = from_f32<T>(dmu);
          out[row * a.ld_out + D + d] = from_f32<T>(dlv);
        }
      }
    }
  }
}

// ---- vectorised kernels for the common geometry: T (threads of the emulated ATen launch) a multiple of `latent`, latent
// even.  Work item q = (m, i): the four rows r0 + j*R (R = T / latent, r0 = 4*m*R + i) share their Philox outputs: element
// (row r0 + j*R, d) is component j of call m of "thread" i*latent + d -- no division per element.  A lane owns TWO
// adjacent features: 4-byte loads of the 16-bit inputs (8-byte for fp32), 8-byte stores -> every warp request is a
// full 128 / 256-byte line.
// Resident blocks per SM the vectorised kernels are compiled for (register cap 64); 3 / 5 / 6 blocks per SM were
// slower (DESIGN.md section 4.4).
constexpr int kBnVecBlocks = 4;
template <typename T> struct Pair;
template <> struct Pair<float> {
  __device__ static __forceinline__ float2 load(const float* p) { return *reinterpret_cast<const float2*>(p); }
  __device__ static __forceinline__ void store(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
};
template <> struct Pair<__nv_bfloat16> {
  __device__ static __forceinline__ float2 load(const __nv_bfloat16* p) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
  }
  __device__ static __forceinline__ void store(__nv_bfloat16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __nv_bfloat162(__float2bfloat16_rn(a), __float2bfloat16_rn(b));
  }
};
template <> struct Pair<__half> {
  __device__ static __forceinline__ float2 load(const __half* p) { return __half22float2(*reinterpret_cast<const __half2*>(p)); }
  __device__ static __forceinline__ void store(__half* p, float a, float b) {
    *reinterpret_cast<__half2*>(p) = __half2(__float2half_rn(a), __float2half_rn(b));
  }
};

__device__ __forceinline__ float comp4(const float4& v, int j) { return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w; }

template <typename T>
__global__ void __launch_bounds__(kBnThreads, kBnVecBlocks) bottleneck_fwd_vec_kernel(BnFwdArgs a) {
  a.pp = resolve(a.pp);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_per_block = kBnThreads / 32;
  const T* __restrict__ in = reinterpret_cast<const T*>(a.mulogvar);
  const int D = a.latent;
  const int64_t R = a.rows_per_T;
  float block_part = 0.f;

  for (int64_t q = (int64_t)blockIdx.x * warps_per_block + warp; q < a.quads; q += (int64_t)gridDim.x * warps_per_block) {
    const int64_t m = q / R, i = q - m * R;
    const int64_t r0 = 4 * m * R + i;
    float rowsum[4] = {0.f, 0.f, 0.f, 0.f};
    for (int d = 2 * lane; d < D; d += 64) {
      const float4 na = normal4_at(a.pp, i * D + d, m), nb = normal4_at(a.pp, i * D + d + 1, m);
      float2 mu[4], lv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {                      // all loads first: eight 128-byte requests in flight per warp
        const int64_t row = r0 + j * R;
        if (row < a.rows) {
          mu[j] = Pair<T>::load(in + row * a.ld + d);
          lv[j] = Pair<T>::load(in + row * a.ld + D + d);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t row = r0 + j * R;
        if (row < a.rows) {
          const float e0 = round_through<T>(comp4(na, j)), e1 = round_through<T>(comp4(nb, j));
          const float v0 = expf(lv[j].x), v1 = expf(lv[j].y);
          const float s0 = sqrtf(v0), s1 = sqrtf(v1);
          // separate roundings (no FMA) so z and kl match the op-by-op torch evaluation bit for bit
          const float z0 = __fadd_rn(mu[j].x, __fmul_rn(e0, s0)), z1 = __fadd_rn(mu[j].y, __fmul_rn(e1, s1));
          const float k0 = __fmul_rn(0.5f, __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(mu[j].x, mu[j].x), v0), lv[j].x), -1.0f));
          const float k1 = __fmul_rn(0.5f, __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(mu[j].y, mu[j].y), v1), lv[j].y), -1.0f));
          const int64_t o = row * D + d;
          Pair<float>::store(a.z + o, z0, z1);
          Pair<float>::store(a.sigma + o, s0, s1);
          if (a.kl_elem) Pair<float>::store(a.kl_elem + o, k0, k1);
          rowsum[j] += k0;                               // (per-lane order d, d + 1: the row sum may differ from the scalar kernel in the last bits)
          rowsum[j] += k1;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t row = r0 + j * R;
      if (row < a.rows) {
        float s = rowsum[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
          a.raw_kl[row] = s;
          block_part += s / (float)a.token_counts[row];
        }
      }
    }
  }

  // deterministic two-level reduction of kl = mean_b(raw_kl[b] / token_counts[b])
  __shared__ float warp_part[kBnThreads / 32];
  __shared__ bool is_last;
  if (lane == 0) warp_part[warp] = block_part;
  __syncthreads();
  unsigned* counter = reinterpret_cast<unsigned*>(a.workspace);
  float* partials = a.workspace + kBnPartialOffset;
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < warps_per_block; ++w) s += warp_part[w];
    partials[blockIdx.x] = s;
    __threadfence();
    unsigned prev = atomicAdd(counter, 1u);
    is_last = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && warp == 0) {
    __threadfence();
    float s = 0.f;
    for (int i = lane; i < (int)gridDim.x; i += 32) s += __ldcg(partials + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      a.kl[0] = s / (float)a.rows;
      *counter = 0u;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kBnThreads, kBnVecBlocks) bottleneck_bwd_vec_kernel(BnBwdArgs a) {
  a.pp = resolve(a.pp);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_per_block = kBnThreads / 32;
  const T* __restrict__ in = reinterpret_cast<const T*>(a.mulogvar);
  T* __restrict__ out = reinterpret_cast<T*>(a.dout);
  const int D = a.latent;
  const int64_t R = a.rows_per_T;
  const float dkl = a.dkl ? a.dkl[0] : 0.f;

  for (int64_t q = (int64_t)blockIdx.x * warps_per_block + warp; q < a.quads; q += (int64_t)gridDim.x * warps_per_block) {
    const int64_t m = q / R, i = q - m * R;
    const int64_t r0 = 4 * m * R + i;
    for (int d = 2 * lane; d < D; d += 64) {
      const float4 na = normal4_at(a.pp, i * D + d, m), nb = normal4_at(a.pp, i * D + d + 1, m);
      float2 mu[4], lv[4], gz[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t row = r0 + j * R;
        if (row < a.rows) {
          mu[j] = Pair<T>::load(in + row * a.ld + d);
          lv[j] = Pair<T>::load(in + row * a.ld + D + d);
          gz[j] = a.dz ? Pair<float>::load(a.dz + row * D + d) : make_float2(0.f, 0.f);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t row = r0 + j * R;
        if (row < a.rows) {
          const int64_t o = row * D + d;
          const float e0 = round_through<T>(comp4(na, j)), e1 = round_through<T>(comp4(nb, j));
          const float v0 = expf(lv[j].x), v1 = expf(lv[j].y);
          const float s0 = sqrtf(v0), s1 = sqrtf(v1);
          float g = dkl / ((float)a.rows * (float)a.token_counts[row]);
          if (a.draw_kl) g += a.draw_kl[row];
          float g0 = g, g1 = g, gs0 = 0.f, gs1 = 0.f;
          if (a.dkl_elem) { const float2 t = Pair<float>::load(a.dkl_elem + o); g0 += t.x; g1 += t.y; }
          if (a.dsigma) { const float2 t = Pair<float>::load(a.dsigma + o); gs0 = t.x; gs1 = t.y; }
          const float dmu0 = gz[j].x + g0 * mu[j].x, dmu1 = gz[j].y + g1 * mu[j].y;
          const float dlv0 = (gz[j].x * e0 + gs0) * 0.5f * s0 + g0 * 0.5f * (v0 - 1.0f);
          const float dlv1 = (gz[j].y * e1 + gs1) * 0.5f * s1 + g1 * 0.5f * (v1 - 1.0f);
          Pair<T>::store(out + row * a.ld_out + d, dmu0, dmu1);
          Pair<T>::store(out + row * a.ld_out + D + d, dlv0, dlv1);
        }
      }
    }
  }
}

struct BnPlan {
  PhiloxPlan pp;
  bool share;
  bool vec;        // the vectorised kernels apply (share, even latent; alignment is checked per call)
  int64_t quads, rows_per_T;
  int grid;
};

static int make_plan(int64_t rows, int latent, uint64_t seed, uint64_t offset, int sm_count, int max_threads_per_sm,
                     BnPlan* p) {
  SVAE_REQUIRE(rows > 0 && latent > 0, SVAE_ERR_INVALID, "bottleneck: rows (%lld) and latent (%d) must be positive",
               (long long)rows, latent);
  SVAE_REQUIRE(offset % 4 == 0, SVAE_ERR_INVALID, "bottleneck: Philox offset %llu is not a multiple of 4",
               (unsigned long long)offset);
  SVAE_REQUIRE(sm_count > 0 && max_threads_per_sm >= 256, SVAE_ERR_INVALID, "bottleneck: bad device geometry");
  int64_t numel = rows * latent;
  int64_t T = 256 * aten_grid(numel, sm_count, max_threads_per_sm);
  p->pp.seed = seed;
  p->pp.offset = offset;
  p->pp.T = T;
  p->pp.dev = nullptr;
  p->share = (T % latent == 0);
  p->vec = p->share && latent % 2 == 0;
  if (p->share) {
    int64_t R = T / latent;
    p->rows_per_T = R;
    p->quads = (rows / (4 * R)) * R + ((rows % (4 * R)) < R ? (rows % (4 * R)) : R);
  } else {
    p->rows_per_T = 1;
    p->quads = rows;
  }
  int64_t blocks = (p->quads + (kBnThreads / 32) - 1) / (kBnThreads / 32);
  int64_t cap = (int64_t)sm_count * 8 < kBnMaxBlocks ? (int64_t)sm_count * 8 : kBnMaxBlocks;
  p->grid = (int)(blocks < cap ? blocks : cap);
  return SVAE_OK;
}

}  // namespace svae

using namespace svae;

extern "C" uint64_t svae_bottleneck_philox_increment(int64_t rows, int32_t latent, int32_t sm_count,
                                                     int32_t max_threads_per_sm) {
  int64_t numel = rows * (int64_t)latent;
  if (numel <= 0 || sm_count <= 0 || max_threads_per_sm < 256) return 0;
  int64_t grid = aten_grid(numel, sm_count, max_threads_per_sm);
  return (uint64_t)(((numel - 1) / (256 * grid * 4) + 1) * 4);
}

extern "C" int svae_bottleneck_fwd_g(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                                     int64_t rows, int32_t latent, uint64_t seed, uint64_t offset, const uint64_t* philox_dev,
                                     int32_t sm_count, int32_t max_threads_per_sm, float* z, float* sigma, float* kl_elem,
                                     float* raw_kl, float* kl, void* workspace, void* stream) {
  SVAE_REQUIRE(mulogvar && token_counts && z && sigma && raw_kl && kl && workspace, SVAE_ERR_INVALID,
               "svae_bottleneck_fwd: null pointer argument");
  SVAE_REQUIRE(ld >= 2 * (int64_t)latent, SVAE_ERR_INVALID, "svae_bottleneck_fwd: ld (%lld) < 2*latent (%d)",
               (long long)ld, 2 * latent);
  BnPlan p;
  int rc = make_plan(rows, latent, seed, offset, sm_count, max_threads_per_sm, &p);
  if (rc) return rc;
  p.pp.dev = philox_dev;
  BnFwdArgs a{mulogvar, ld, token_counts, rows, latent, p.pp, z, sigma, kl_elem, raw_kl, kl,
              reinterpret_cast<float*>(workspace), p.quads, p.rows_per_T};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ScopedKernelTimer timer("bottleneck_fwd", st);
  // 4 / 8-byte accesses of the vectorised kernel: even leading dimension, aligned bases
  const size_t es = dtype_size(dtype);
  const bool vec = p.vec && ld % 2 == 0 && reinterpret_cast<uintptr_t>(mulogvar) % (2 * es) == 0 &&
                   reinterpret_cast<uintptr_t>(z) % 8 == 0 && reinterpret_cast<uintptr_t>(sigma) % 8 == 0 &&
                   reinterpret_cast<uintptr_t>(kl_elem) % 8 == 0;
#define SVAE_BN_LAUNCH(T)                                                              \
  do {                                                                                 \
    if (vec) bottleneck_fwd_vec_kernel<T><<<p.grid, kBnThreads, 0, st>>>(a);           \
    else if (p.share) bottleneck_fwd_kernel<T, true><<<p.grid, kBnThreads, 0, st>>>(a); \
    else bottleneck_fwd_kernel<T, false><<<p.grid, kBnThreads, 0, st>>>(a);            \
  } while (0)
  switch (dtype) {
    case SVAE_DTYPE_F32: SVAE_BN_LAUNCH(float); break;
    case SVAE_DTYPE_BF16: SVAE_BN_LAUNCH(__nv_bfloat16); break;
    case SVAE_DTYPE_F16: SVAE_BN_LAUNCH(__half); break;
    default: SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_bottleneck_fwd: unknown dtype %d", dtype);
  }
#undef SVAE_BN_LAUNCH
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

extern "C" int svae_bottleneck_fwd(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                                   int64_t rows, int32_t latent, uint64_t seed, uint64_t offset, int32_t sm_count,
                                   int32_t max_threads_per_sm, float* z, float* sigma, float* kl_elem, float* raw_kl,
                                   float* kl, void* workspace, void* stream) {
  return svae_bottleneck_fwd_g(mulogvar, ld, dtype, token_counts, rows, latent, seed, offset, nullptr, sm_count, max_threads_per_sm, z,
                               sigma, kl_elem, raw_kl, kl, workspace, stream);
}

extern "C" int svae_bottleneck_bwd_g(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                                     int64_t rows, int32_t latent, uint64_t seed, uint64_t offset, const uint64_t* philox_dev,
                                     int32_t sm_count, int32_t max_threads_per_sm, const float* dz, const float* dsigma,
                                     const float* dkl_elem, const float* draw_kl, const float* dkl, void* d_mulogvar,
                                     int64_t ld_out, void* stream) {
  SVAE_REQUIRE(mulogvar && token_counts && d_mulogvar, SVAE_ERR_INVALID, "svae_bottleneck_bwd: null pointer argument");
  SVAE_REQUIRE(ld >= 2 * (int64_t)latent && ld_out >= 2 * (int64_t)latent, SVAE_ERR_INVALID,
               "svae_bottleneck_bwd: leading dimension smaller than 2*latent");
  BnPlan p;
  int rc = make_plan(rows, latent, seed, offset, sm_count, max_threads_per_sm, &p);
  if (rc) return rc;
  p.pp.dev = philox_dev;
  BnBwdArgs a{mulogvar, ld, token_counts, rows, latent, p.pp, dz, dsigma, dkl_elem, draw_kl, dkl, d_mulogvar, ld_out,
              p.quads, p.rows_per_T};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ScopedKernelTimer timer("bottleneck_bwd", st);
  const size_t es = dtype_size(dtype);
  const bool vec = p.vec && ld % 2 == 0 && ld_out % 2 == 0 && reinterpret_cast<uintptr_t>(mulogvar) % (2 * es) == 0 &&
                   reinterpret_cast<uintptr_t>(d_mulogvar) % (2 * es) == 0 && reinterpret_cast<uintptr_t>(dz) % 8 == 0 &&
                   reinterpret_cast<uintptr_t>(dsigma) % 8 == 0 && reinterpret_cast<uintptr_t>(dkl_elem) % 8 == 0;
#define SVAE_BN_LAUNCH(T)                                                              \
  do {                                                                                 \
    if (vec) bottleneck_bwd_vec_kernel<T><<<p.grid, kBnThreads, 0, st>>>(a);           \
    else if (p.share) bottleneck_bwd_kernel<T, true><<<p.grid, kBnThreads, 0, st>>>(a); \
    else bottleneck_bwd_kernel<T, false><<<p.grid, kBnThreads, 0, st>>>(a);            \
  } while (0)
  switch (dtype) {
    case SVAE_DTYPE_F32: SVAE_BN_LAUNCH(float); break;
    case SVAE_DTYPE_BF16: SVAE_BN_LAUNCH(__nv_bfloat16); break;
    case SVAE_DTYPE_F16: SVAE_BN_LAUNCH(__half); break;
    default: SVAE_REQUIRE(false, SVAE_ERR_INVALID, "svae_bottleneck_bwd: unknown dtype %d", dtype);
  }
#undef SVAE_BN_LAUNCH
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

extern "C" int svae_bottleneck_bwd(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                                   int64_t rows, int32_t latent, uint64_t seed, uint64_t offset, int32_t sm_count,
                                   int32_t max_threads_per_sm, const float* dz, const float* dsigma,
                                   const float* dkl_elem, const float* draw_kl, const float* dkl, void* d_mulogvar,
                                   int64_t ld_out, void* stream) {
  return svae_bottleneck_bwd_g(mulogvar, ld, dtype, token_counts, rows, latent, seed, offset, nullptr, sm_count, max_threads_per_sm, dz,
                               dsigma, dkl_elem, draw_kl, dkl, d_mulogvar, ld_out, stream);
}
