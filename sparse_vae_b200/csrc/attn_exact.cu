// Exact (fp32 FFMA, CUDA-core) block-sparse attention forward/backward.
//
// This is the PARITY MODE of the path: fp32 inputs cannot meet the reference's 1e-4 bound on TF32 tensor cores
// (10-bit mantissa), so fp32 tensors run here; 16-bit inputs can be forced through it (SVAE_ATTN_FORCE_EXACT) to
// cross-check the tcgen05 kernels on the device.  It is not the performance path.
//
// Algorithm per 32-row query block r (reference core/sparse_attention.py:75-92, restated block by block):
//   for every live key block c of block-row r (band + optional global column 0):
//       S = Q_r K_c^T * scale + kpm[key] ; causal: key > query -> -inf        (sdd + softmax prologue)
//       online softmax update (m, l) ; O += P V_c                              (softmax + dsd)
//   O /= l ; lse = m + log l
// Backward per query block (reference core/sparse_matmul.py:463-488 + softmax backward):
//   P = exp(S - lse), dP = dO V_c^T, dS = P*(dP - rowsum(dO*O))*scale,
//   dQ_r += dS K_c (registers), dK_c += dS^T Q_r, dV_c += P^T dO_r (fp32 atomics into the workspace).
#include <math.h>

#include "common.cuh"

namespace svae {

constexpr int kBlk = 32;
constexpr int kExThreads = 128;

struct ExactArgs {
  const void *q, *k, *v, *o, *dout;
  const float* kpm;
  const float* lse_in;
  void* out;
  float* lse;
  void* dq;
  float *dk_acc, *dv_acc;   // fp32 [B,H,L,Dh] contiguous accumulators (backward)
  int B, H, L, Dh, nb;
  Band band;
  int causal;
  float scale;
  int64_t qs[3], ks[3], vs[3], os[3], dos[3], dqs[3];
};

template <typename T>
__device__ __forceinline__ void load_tile(float* dst, int ld, const T* src, int64_t row_stride, int row0, int L,
                                          int Dh) {
  // 32 rows x Dh, coalesced along Dh
  for (int i = threadIdx.x; i < kBlk * Dh; i += kExThreads) {
    int r = i / Dh, c = i - r * Dh;
    float val = 0.f;
    if (row0 + r < L) val = to_f32<T>(src[(int64_t)(row0 + r) * row_stride + c]);
    dst[r * ld + c] = val;
  }
}

// live key blocks of block-row r in ascending order: returns count, fills list
__device__ __forceinline__ int live_blocks(const Band& g, int r, int nb, int* list) {
  int n = 0;
  int lo = r - (g.left - 1), hi = r + g.nsup;
  if (lo < 0) lo = 0;
  if (hi > nb - 1) hi = nb - 1;
  if (g.cls && lo > 0) list[n++] = 0;
  for (int c = lo; c <= hi; ++c) list[n++] = c;
  return n;
}

constexpr int kMaxLive = 64;

template <typename T, int DH>
__global__ void __launch_bounds__(kExThreads) attn_exact_fwd_kernel(ExactArgs a) {
  constexpr int LD = DH + 1;
  // head 128: the tiles exceed 48 KB of static shared memory and live in the dynamic allocation instead
  constexpr bool kDyn = DH > 64;
  __shared__ float Qs_[kDyn ? 1 : kBlk * LD], Ks_[kDyn ? 1 : kBlk * LD], Vs_[kDyn ? 1 : kBlk * LD],
      Ps_[kDyn ? 1 : kBlk * (kBlk + 1)];
  extern __shared__ float dyn_tiles[];
  float* Qs = kDyn ? dyn_tiles : Qs_;
  float* Ks = kDyn ? dyn_tiles + kBlk * LD : Ks_;
  float* Vs = kDyn ? dyn_tiles + 2 * kBlk * LD : Vs_;
  float* Ps = kDyn ? dyn_tiles + 3 * kBlk * LD : Ps_;
  __shared__ float kpm_s[kBlk];
  __shared__ int live[kMaxLive];
  __shared__ int nlive;

  const int r = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x;
  const int row = tid >> 2, sub = tid & 3;
  const T* q = reinterpret_cast<const T*>(a.q) + b * a.qs[0] + h * a.qs[1];
  const T* k = reinterpret_cast<const T*>(a.k) + b * a.ks[0] + h * a.ks[1];
  const T* v = reinterpret_cast<const T*>(a.v) + b * a.vs[0] + h * a.vs[1];

  if (tid == 0) nlive = live_blocks(a.band, r, a.nb, live);
  load_tile<T>(Qs, LD, q, a.qs[2], r * kBlk, a.L, DH);
  __syncthreads();

  float m = -INFINITY, l = 0.f;
  float acc[DH / 4];
#pragma unroll
  for (int i = 0; i < DH / 4; ++i) acc[i] = 0.f;

  const int n = nlive;
  for (int it = 0; it < n; ++it) {
    const int c = live[it];
    __syncthreads();   // previous iteration done with Ks/Vs/Ps
    load_tile<T>(Ks, LD, k, a.ks[2], c * kBlk, a.L, DH);
    load_tile<T>(Vs, LD, v, a.vs[2], c * kBlk, a.L, DH);
    if (tid < kBlk) kpm_s[tid] = a.kpm ? a.kpm[(int64_t)b * a.L + c * kBlk + tid] : 0.f;
    __syncthreads();

    float s[8];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = sub + 4 * j;
      float d = 0.f;
#pragma unroll 8
      for (int e = 0; e < DH; ++e) d = fmaf(Qs[row * LD + e], Ks[col * LD + e], d);
      d = d * a.scale + kpm_s[col];
      if (a.causal && (c * kBlk + col > r * kBlk + row)) d = -INFINITY;
      s[j] = d;
      mx = fmaxf(mx, d);
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float m_new = fmaxf(m, mx);
    const float m_safe = (m_new == -INFINITY) ? 0.f : m_new;
    const float alpha = (m == -INFINITY) ? 0.f : expf(m - m_safe);
    float ps = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float p = expf(s[j] - m_safe);      // exp(-inf) = 0
      Ps[row * (kBlk + 1) + sub + 4 * j] = p;
      ps += p;
    }
    ps += __shfl_xor_sync(0xffffffffu, ps, 1);
    ps += __shfl_xor_sync(0xffffffffu, ps, 2);
    l = l * alpha + ps;
    m = m_new;
#pragma unroll
    for (int i = 0; i < DH / 4; ++i) acc[i] *= alpha;
    __syncwarp();   // the 4 threads of a row are in the same warp; Ps rows are warp-private
#pragma unroll 4
    for (int key = 0; key < kBlk; ++key) {
      const float p = Ps[row * (kBlk + 1) + key];
#pragma unroll
      for (int i = 0; i < DH / 4; ++i) acc[i] = fmaf(p, Vs[key * LD + sub + 4 * i], acc[i]);
    }
  }

  const int qrow = r * kBlk + row;
  if (qrow < a.L) {
    T* o = reinterpret_cast<T*>(a.out) + b * a.os[0] + h * a.os[1] + (int64_t)qrow * a.os[2];
    const float inv = 1.0f / l;          // l == 0 (fully masked row) -> NaN like the reference softmax
#pragma unroll
    for (int i = 0; i < DH / 4; ++i) o[sub + 4 * i] = from_f32<T>(acc[i] * inv);
    if (sub == 0) a.lse[((int64_t)b * a.H + h) * a.L + qrow] = m + logf(l);
  }
}

template <typename T, int DH>
__global__ void __launch_bounds__(kExThreads) attn_exact_bwd_kernel(ExactArgs a) {
  constexpr int LD = DH + 1;
  constexpr bool kDyn = DH > 64;                      // see attn_exact_fwd_kernel
  __shared__ float Qs_[kDyn ? 1 : kBlk * LD], Ks_[kDyn ? 1 : kBlk * LD], Vs_[kDyn ? 1 : kBlk * LD],
      dOs_[kDyn ? 1 : kBlk * LD];
  __shared__ float Ps_[kDyn ? 1 : kBlk * (kBlk + 1)], dSs_[kDyn ? 1 : kBlk * (kBlk + 1)];
  extern __shared__ float dyn_tiles[];
  float* Qs = kDyn ? dyn_tiles : Qs_;
  float* Ks = kDyn ? dyn_tiles + kBlk * LD : Ks_;
  float* Vs = kDyn ? dyn_tiles + 2 * kBlk * LD : Vs_;
  float* dOs = kDyn ? dyn_tiles + 3 * kBlk * LD : dOs_;
  float* Ps = kDyn ? dyn_tiles + 4 * kBlk * LD : Ps_;
  float* dSs = kDyn ? dyn_tiles + 4 * kBlk * LD + kBlk * (kBlk + 1) : dSs_;
  __shared__ float kpm_s[kBlk];
  __shared__ int live[kMaxLive];
  __shared__ int nlive;

  const int r = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x;
  const int row = tid >> 2, sub = tid & 3;
  const T* q = reinterpret_cast<const T*>(a.q) + b * a.qs[0] + h * a.qs[1];
  const T* k = reinterpret_cast<const T*>(a.k) + b * a.ks[0] + h * a.ks[1];
  const T* v = reinterpret_cast<const T*>(a.v) + b * a.vs[0] + h * a.vs[1];
  const T* o = reinterpret_cast<const T*>(a.o) + b * a.os[0] + h * a.os[1];
  const T* dO = reinterpret_cast<const T*>(a.dout) + b * a.dos[0] + h * a.dos[1];

  if (tid == 0) nlive = live_blocks(a.band, r, a.nb, live);
  load_tile<T>(Qs, LD, q, a.qs[2], r * kBlk, a.L, DH);
  load_tile<T>(dOs, LD, dO, a.dos[2], r * kBlk, a.L, DH);
  __syncthreads();

  const int qrow = r * kBlk + row;
  // delta = rowsum(dO * O); each of the 4 threads of a row sums a quarter
  float delta = 0.f;
  if (qrow < a.L) {
    for (int e = sub; e < DH; e += 4) delta += dOs[row * LD + e] * to_f32<T>(o[(int64_t)qrow * a.os[2] + e]);
  }
  delta += __shfl_xor_sync(0xffffffffu, delta, 1);
  delta += __shfl_xor_sync(0xffffffffu, delta, 2);
  const float lse = (qrow < a.L) ? a.lse_in[((int64_t)b * a.H + h) * a.L + qrow] : 0.f;

  float dq[DH / 4];
#pragma unroll
  for (int i = 0; i < DH / 4; ++i) dq[i] = 0.f;

  const int n = nlive;
  for (int it = 0; it < n; ++it) {
    const int c = live[it];
    __syncthreads();
    load_tile<T>(Ks, LD, k, a.ks[2], c * kBlk, a.L, DH);
    load_tile<T>(Vs, LD, v, a.vs[2], c * kBlk, a.L, DH);
    if (tid < kBlk) kpm_s[tid] = a.kpm ? a.kpm[(int64_t)b * a.L + c * kBlk + tid] : 0.f;
    __syncthreads();

#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = sub + 4 * j;
      float s = 0.f, dp = 0.f;
#pragma unroll 8
      for (int e = 0; e < DH; ++e) {
        s = fmaf(Qs[row * LD + e], Ks[col * LD + e], s);
        dp = fmaf(dOs[row * LD + e], Vs[col * LD + e], dp);
      }
      s = s * a.scale + kpm_s[col];
      if (a.causal && (c * kBlk + col > qrow)) s = -INFINITY;
      float p = (qrow < a.L && c * kBlk + col < a.L) ? expf(s - lse) : 0.f;
      if (s == -INFINITY) p = 0.f;   // also covers lse == -inf rows
      Ps[row * (kBlk + 1) + col] = p;
      dSs[row * (kBlk + 1) + col] = p * (dp - delta) * a.scale;
    }
    __syncthreads();

    // dQ_r += dS K_c
#pragma unroll 4
    for (int key = 0; key < kBlk; ++key) {
      const float ds = dSs[row * (kBlk + 1) + key];
#pragma unroll
      for (int i = 0; i < DH / 4; ++i) dq[i] = fmaf(ds, Ks[key * LD + sub + 4 * i], dq[i]);
    }
    // dV_c += P^T dO_r ; dK_c += dS^T Q_r  (thread: key = row index here, columns sub + 4 i)
    {
      const int key = row;
      float dv[DH / 4], dk[DH / 4];
#pragma unroll
      for (int i = 0; i < DH / 4; ++i) dv[i] = dk[i] = 0.f;
#pragma unroll 4
      for (int rr = 0; rr < kBlk; ++rr) {
        const float p = Ps[rr * (kBlk + 1) + key];
        const float ds = dSs[rr * (kBlk + 1) + key];
#pragma unroll
        for (int i = 0; i < DH / 4; ++i) {
          dv[i] = fmaf(p, dOs[rr * LD + sub + 4 * i], dv[i]);
          dk[i] = fmaf(ds, Qs[rr * LD + sub + 4 * i], dk[i]);
        }
      }
      const int krow = c * kBlk + key;
      if (krow < a.L) {
        const int64_t base = (((int64_t)b * a.H + h) * a.L + krow) * DH;
#pragma unroll
        for (int i = 0; i < DH / 4; ++i) {
          atomicAdd(a.dv_acc + base + sub + 4 * i, dv[i]);
          atomicAdd(a.dk_acc + base + sub + 4 * i, dk[i]);
        }
      }
    }
  }

  if (qrow < a.L) {
    T* dqp = reinterpret_cast<T*>(a.dq) + b * a.dqs[0] + h * a.dqs[1] + (int64_t)qrow * a.dqs[2];
#pragma unroll
    for (int i = 0; i < DH / 4; ++i) dqp[sub + 4 * i] = from_f32<T>(dq[i]);
  }
}

// fp32 contiguous [B,H,L,Dh] accumulator -> strided output of dtype T
template <typename T>
__global__ void convert_out_kernel(const float* __restrict__ src, T* __restrict__ dst, int64_t total, int H, int L,
                                   int Dh, int64_t s0, int64_t s1, int64_t s2) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int d = (int)(i % Dh);
    int64_t t = i / Dh;
    int l = (int)(t % L);
    t /= L;
    int h = (int)(t % H);
    int64_t b = t / H;
    dst[b * s0 + h * s1 + (int64_t)l * s2 + d] = from_f32<T>(src[i]);
  }
}

static void fill_args(ExactArgs& a, const svae_attn_desc* d) {
  a.B = d->batch; a.H = d->heads; a.L = d->seq_len; a.Dh = d->head_dim;
  a.nb = d->seq_len / d->block_size;
  a.band = make_band(d->window_size, d->causal, d->include_cls);
  a.causal = d->causal;
  a.scale = d->scale;
  for (int i = 0; i < 3; ++i) {
    a.qs[i] = d->q_stride[i]; a.ks[i] = d->k_stride[i]; a.vs[i] = d->v_stride[i]; a.os[i] = d->o_stride[i];
    a.dos[i] = d->do_stride[i]; a.dqs[i] = d->dq_stride[i];
  }
}

template <typename T>
static int launch_fwd_t(const ExactArgs& a, cudaStream_t st) {
  dim3 grid(a.nb, a.H, a.B);
  ScopedKernelTimer timer("attn_exact_fwd", st);
  switch (a.Dh) {
    case 16: attn_exact_fwd_kernel<T, 16><<<grid, kExThreads, 0, st>>>(a); break;
    case 32: attn_exact_fwd_kernel<T, 32><<<grid, kExThreads, 0, st>>>(a); break;
    case 64: attn_exact_fwd_kernel<T, 64><<<grid, kExThreads, 0, st>>>(a); break;
    case 128: {
      constexpr int bytes = (3 * kBlk * 129 + kBlk * (kBlk + 1)) * 4;
      auto kern = attn_exact_fwd_kernel<T, 128>;
      SVAE_CONFIGURE_SMEM(kern, bytes);
      kern<<<grid, kExThreads, bytes, st>>>(a);
      break;
    }
    default: SVAE_REQUIRE(false, SVAE_ERR_UNSUPPORTED, "exact attention: head_dim %d not in {16,32,64,128}", a.Dh);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

template <typename T>
static int launch_bwd_t(const ExactArgs& a, const svae_attn_desc* d, void* dk, void* dv, cudaStream_t st) {
  dim3 grid(a.nb, a.H, a.B);
  const int64_t total = (int64_t)a.B * a.H * a.L * a.Dh;
  SVAE_CUDA_CHECK(cudaMemsetAsync(a.dk_acc, 0, sizeof(float) * total * 2, st));   // dk_acc and dv_acc are adjacent
  ScopedKernelTimer timer("attn_exact_bwd", st);
  switch (a.Dh) {
    case 16: attn_exact_bwd_kernel<T, 16><<<grid, kExThreads, 0, st>>>(a); break;
    case 32: attn_exact_bwd_kernel<T, 32><<<grid, kExThreads, 0, st>>>(a); break;
    case 64: attn_exact_bwd_kernel<T, 64><<<grid, kExThreads, 0, st>>>(a); break;
    case 128: {
      constexpr int bytes = (4 * kBlk * 129 + 2 * kBlk * (kBlk + 1)) * 4;
      auto kern = attn_exact_bwd_kernel<T, 128>;
      SVAE_CONFIGURE_SMEM(kern, bytes);
      kern<<<grid, kExThreads, bytes, st>>>(a);
      break;
    }
    default: SVAE_REQUIRE(false, SVAE_ERR_UNSUPPORTED, "exact attention: head_dim %d not in {16,32,64,128}", a.Dh);
  }
  SVAE_CUDA_CHECK(cudaGetLastError());
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  convert_out_kernel<T><<<blocks, 256, 0, st>>>(a.dk_acc, reinterpret_cast<T*>(dk), total, a.H, a.L, a.Dh,
                                                d->dk_stride[0], d->dk_stride[1], d->dk_stride[2]);
  convert_out_kernel<T><<<blocks, 256, 0, st>>>(a.dv_acc, reinterpret_cast<T*>(dv), total, a.H, a.L, a.Dh,
                                                d->dv_stride[0], d->dv_stride[1], d->dv_stride[2]);
  SVAE_CUDA_CHECK(cudaGetLastError());
  return SVAE_OK;
}

int exact_fwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm, void* out,
              float* lse, cudaStream_t st) {
  SVAE_REQUIRE(make_band(d->window_size, d->causal, d->include_cls).left +
                       make_band(d->window_size, d->causal, d->include_cls).nsup + 1 <= kMaxLive,
               SVAE_ERR_UNSUPPORTED, "exact attention: window_size %d too large", d->window_size);
  ExactArgs a{};
  fill_args(a, d);
  a.q = q; a.k = k; a.v = v; a.kpm = kpm; a.out = out; a.lse = lse;
  switch (d->dtype) {
    case SVAE_DTYPE_F32: return launch_fwd_t<float>(a, st);
    case SVAE_DTYPE_BF16: return launch_fwd_t<__nv_bfloat16>(a, st);
    case SVAE_DTYPE_F16: return launch_fwd_t<__half>(a, st);
  }
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "unknown dtype %d", d->dtype);
}

size_t exact_bwd_workspace(const svae_attn_desc* d) {
  return sizeof(float) * 2 * (size_t)d->batch * d->heads * d->seq_len * d->head_dim;
}

int exact_bwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out, const void* dout,
              const float* lse, const float* kpm, void* dq, void* dk, void* dv, void* workspace, cudaStream_t st) {
  SVAE_REQUIRE(make_band(d->window_size, d->causal, d->include_cls).left +
                       make_band(d->window_size, d->causal, d->include_cls).nsup + 1 <= kMaxLive,
               SVAE_ERR_UNSUPPORTED, "exact attention: window_size %d too large", d->window_size);
  ExactArgs a{};
  fill_args(a, d);
  a.q = q; a.k = k; a.v = v; a.o = out; a.dout = dout; a.kpm = kpm; a.lse_in = lse; a.dq = dq;
  const size_t total = (size_t)d->batch * d->heads * d->seq_len * d->head_dim;
  a.dk_acc = reinterpret_cast<float*>(workspace);
  a.dv_acc = a.dk_acc + total;
  switch (d->dtype) {
    case SVAE_DTYPE_F32: return launch_bwd_t<float>(a, d, dk, dv, st);
    case SVAE_DTYPE_BF16: return launch_bwd_t<__nv_bfloat16>(a, d, dk, dv, st);
    case SVAE_DTYPE_F16: return launch_bwd_t<__half>(a, d, dk, dv, st);
  }
  SVAE_REQUIRE(false, SVAE_ERR_INVALID, "unknown dtype %d", d->dtype);
}

}  // namespace svae
