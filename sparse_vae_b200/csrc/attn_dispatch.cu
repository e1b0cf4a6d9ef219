// C-ABI entry points of the attention path: argument validation, TMA descriptor encoding, path selection.
//   fp32 tensors (or SVAE_ATTN_FORCE_EXACT)  -> exact CUDA-core kernels (attn_exact.cu)   [parity mode]
//   bf16 / fp16 tensors                      -> tcgen05 / TMEM / TMA kernels (attn_*_sm100.cu)
#include <mutex>

#include "attn_sm100.cuh"

namespace svae {

int exact_fwd(const svae_attn_desc*, const void*, const void*, const void*, const float*, void*, float*, cudaStream_t);
size_t exact_bwd_workspace(const svae_attn_desc*);
int exact_bwd(const svae_attn_desc*, const void*, const void*, const void*, const void*, const void*, const float*,
              const float*, void*, void*, void*, void*, cudaStream_t);

namespace sm100 {

int fwd(const svae_attn_desc*, const void*, const void*, const void*, const float*, void*, float*, float*, long long*, cudaStream_t);
bool fwd_persist_supported(const svae_attn_desc*);
int fwd_persist(const svae_attn_desc*, const void*, const void*, const void*, const float*, void*, float*, long long*, cudaStream_t);
size_t bwd_workspace(const svae_attn_desc*);
bool bwd_supported(const svae_attn_desc*);
bool bwd1_supported(const svae_attn_desc*);
size_t bwd1_workspace(const svae_attn_desc*);
int bwd1(const svae_attn_desc*, const void*, const void*, const void*, const void*, const void*, const float*,
         const float*, void*, void*, void*, void*, cudaStream_t);
int bwd(const svae_attn_desc*, const void*, const void*, const void*, const void*, const void*, const float*,
        const float*, void*, void*, void*, void*, cudaStream_t);

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    // resolved through the runtime so the library has no link-time dependency on libcuda.so
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 4-D map {Dh, L, H, B} over a strided [B, H, L, Dh] tensor; box = {Dh, box_rows, 1, 1}; swizzle = row bytes.
int encode_tmap(CUtensorMap* map, CUtensorMapDataType dt, const void* base, int Dh, int L, int H, int B,
                const int64_t stride[3], int box_rows) {
  // A tensor map is a pure function of (base, dtype, dims, strides, box): a training step asks for the same handful
  // again and again (the caching allocator hands back the same addresses), so the last few are kept per thread.
  struct Key {
    const void* base; int dt, Dh, L, H, B, box; int64_t s0, s1, s2;
    bool operator==(const Key& o) const {
      return base == o.base && dt == o.dt && Dh == o.Dh && L == o.L && H == o.H && B == o.B && box == o.box && s0 == o.s0 &&
             s1 == o.s1 && s2 == o.s2;
    }
  };
  constexpr int kCache = 64;
  static thread_local Key keys[kCache];
  static thread_local CUtensorMap maps[kCache];
  static thread_local int used = 0, next = 0;
  const Key key{base, (int)dt, Dh, L, H, B, box_rows, stride[0], stride[1], stride[2]};
  for (int i = 0; i < used; ++i)
    if (keys[i] == key) { *map = maps[i]; return SVAE_OK; }
  EncodeTiledFn fn = get_encode_fn();
  SVAE_REQUIRE(fn != nullptr, SVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the CUDA driver");
  // cuTensorMapEncodeTiled is a DRIVER call: on a thread that has not made a runtime call yet (PyTorch's autograd
  // thread entering the backward) no context is current and it fails with CUDA_ERROR_INVALID_CONTEXT
  static thread_local bool context_bound = false;
  if (!context_bound) {
    SVAE_CUDA_CHECK(cudaFree(nullptr));
    context_bound = true;
  }
  const int64_t es = 2;
  cuuint64_t dims[4] = {(cuuint64_t)Dh, (cuuint64_t)L, (cuuint64_t)H, (cuuint64_t)B};
  // a size-1 dimension may carry any stride; give it a harmless, valid one
  int64_t s_row = stride[2], s_head = H > 1 ? stride[1] : (int64_t)Dh, s_batch = B > 1 ? stride[0] : (int64_t)L * stride[2];
  if (L == 1) s_row = Dh;
  cuuint64_t strides[3] = {(cuuint64_t)(s_row * es), (cuuint64_t)(s_head * es), (cuuint64_t)(s_batch * es)};
  cuuint32_t box[4] = {(cuuint32_t)Dh, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const int rowb = Dh * 2;
  CUtensorMapSwizzle sw = rowb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : rowb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                               : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = fn(map, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SVAE_REQUIRE(r == CUDA_SUCCESS, SVAE_ERR_CUDA,
               "cuTensorMapEncodeTiled failed (%d): base=%p dims={%d,%d,%d,%d} strides(elem)={%lld,%lld,%lld}", (int)r,
               base, Dh, L, H, B, (long long)s_row, (long long)s_head, (long long)s_batch);
  keys[next] = key;
  maps[next] = *map;
  next = (next + 1) % kCache;
  if (used < kCache) ++used;
  return SVAE_OK;
}

int encode_tmap_2d(CUtensorMap* map, CUtensorMapDataType dt, const void* base, int64_t cols, int64_t rows, int64_t ld,
                   int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  SVAE_REQUIRE(fn != nullptr, SVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the CUDA driver");
  static thread_local bool context_bound = false;      // see encode_tmap
  if (!context_bound) {
    SVAE_CUDA_CHECK(cudaFree(nullptr));
    context_bound = true;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)((rows > 1 ? ld : cols) * 2)};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SVAE_REQUIRE(r == CUDA_SUCCESS, SVAE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d): base=%p dims={%lld,%lld} ld=%lld",
               (int)r, base, (long long)cols, (long long)rows, (long long)ld);
  return SVAE_OK;
}

}  // namespace sm100

static bool tma_ok(const void* p, const int64_t s[3], int H, int B, int L) {
  if (reinterpret_cast<uintptr_t>(p) % 16) return false;
  if (L > 1 && (s[2] * 2) % 16) return false;
  if (H > 1 && (s[1] * 2) % 16) return false;
  if (B > 1 && (s[0] * 2) % 16) return false;
  return true;
}

static int validate(const svae_attn_desc* d, bool backward) {
  SVAE_REQUIRE(d != nullptr, SVAE_ERR_INVALID, "attention: null descriptor");
  SVAE_REQUIRE(d->batch > 0 && d->heads > 0 && d->seq_len > 0 && d->head_dim > 0, SVAE_ERR_INVALID,
               "attention: non-positive size (B=%d H=%d L=%d Dh=%d)", d->batch, d->heads, d->seq_len, d->head_dim);
  SVAE_REQUIRE(d->block_size == 32, SVAE_ERR_UNSUPPORTED, "attention: block_size %d != 32", d->block_size);
  SVAE_REQUIRE(d->seq_len % d->block_size == 0, SVAE_ERR_INVALID,
               "attention: seq_len %d is not a multiple of the block size %d", d->seq_len, d->block_size);
  SVAE_REQUIRE(d->window_size >= 1, SVAE_ERR_INVALID, "attention: window_size %d < 1", d->window_size);
  SVAE_REQUIRE(d->dtype == SVAE_DTYPE_F32 || d->dtype == SVAE_DTYPE_BF16 || d->dtype == SVAE_DTYPE_F16,
               SVAE_ERR_INVALID, "attention: unknown dtype %d", d->dtype);
  (void)backward;
  return SVAE_OK;
}

static bool use_exact(const svae_attn_desc* d) {
  return d->dtype == SVAE_DTYPE_F32 || (d->flags & SVAE_ATTN_FORCE_EXACT);
}

// one pass over the sequence (attn_bwd1_sm100.cu) unless the geometry is outside it or the caller asks for the
// two-pass kernels (attn_bwd_sm100.cu: non-causal layouts and windows 5..10)
static bool use_one_pass(const svae_attn_desc* d) {
  return !(d->flags & SVAE_ATTN_BWD_TWO_PASS) && sm100::bwd1_supported(d);
}

}  // namespace svae

using namespace svae;

extern "C" int svae_attn_fwd_slots(const svae_attn_desc* d) {
  if (!d || d->block_size <= 0) return -1;
  return sm100::make_geom(d->window_size, d->causal, d->include_cls, d->seq_len / d->block_size).nslots;
}

static int attn_fwd_impl(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm,
                         void* out, float* lse, float* s_dump, long long* timeline, void* stream) {
  int rc = validate(d, false);
  if (rc) return rc;
  SVAE_REQUIRE(q && k && v && out && lse, SVAE_ERR_INVALID, "svae_attn_fwd: null tensor pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (use_exact(d)) {
    SVAE_REQUIRE(s_dump == nullptr, SVAE_ERR_UNSUPPORTED, "score dump is only implemented on the sm100 path");
    return exact_fwd(d, q, k, v, kpm, out, lse, st);
  }
  SVAE_REQUIRE(tma_ok(q, d->q_stride, d->heads, d->batch, d->seq_len) && tma_ok(k, d->k_stride, d->heads, d->batch, d->seq_len) &&
                   tma_ok(v, d->v_stride, d->heads, d->batch, d->seq_len) && tma_ok(out, d->o_stride, d->heads, d->batch, d->seq_len),
               SVAE_ERR_INVALID, "svae_attn_fwd: 16-bit tensors must be 16-byte aligned with strides that are multiples of 8 elements");
  // persistent warp-specialised kernel (69 us vs 104 us at the C2 shape): what the host wrapper asks for whenever the
  // geometry fits (<= 8 key slots); wider windows and score dumps take the one-CTA-per-tile kernel
  if (!s_dump && (d->flags & SVAE_ATTN_PERSISTENT) && sm100::fwd_persist_supported(d))
    return sm100::fwd_persist(d, q, k, v, kpm, out, lse, timeline, st);
  return sm100::fwd(d, q, k, v, kpm, out, lse, s_dump, timeline, st);
}

extern "C" int svae_attn_fwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const float* kpm,
                             void* out, float* lse, void* stream) {
  return attn_fwd_impl(d, q, k, v, kpm, out, lse, nullptr, nullptr, stream);
}

extern "C" int svae_attn_fwd_debug(const svae_attn_desc* d, const void* q, const void* k, const void* v,
                                   const float* kpm, void* out, float* lse, float* s_dump, long long* timeline,
                                   void* stream) {
  return attn_fwd_impl(d, q, k, v, kpm, out, lse, s_dump, timeline, stream);
}

extern "C" size_t svae_attn_bwd_workspace_bytes(const svae_attn_desc* d) {
  if (validate(d, true)) return 0;
  if (use_exact(d) || !sm100::bwd_supported(d)) return exact_bwd_workspace(d);
  if (use_one_pass(d)) return sm100::bwd1_workspace(d);
  return sm100::bwd_workspace(d);
}

extern "C" int svae_attn_bwd_path(const svae_attn_desc* d) {
  if (validate(d, true)) return -1;
  if (use_exact(d) || !sm100::bwd_supported(d)) return SVAE_BWD_PATH_EXACT;
  return use_one_pass(d) ? SVAE_BWD_PATH_TCGEN05 : SVAE_BWD_PATH_TCGEN05_TWO_PASS;
}

extern "C" int svae_attn_bwd(const svae_attn_desc* d, const void* q, const void* k, const void* v, const void* out,
                             const void* dout, const float* lse, const float* kpm, void* dq, void* dk, void* dv,
                             void* workspace, size_t workspace_bytes, void* stream) {
  int rc = validate(d, true);
  if (rc) return rc;
  SVAE_REQUIRE(q && k && v && out && dout && lse && dq && dk && dv && workspace, SVAE_ERR_INVALID,
               "svae_attn_bwd: null pointer argument");
  SVAE_REQUIRE(workspace_bytes >= svae_attn_bwd_workspace_bytes(d), SVAE_ERR_INVALID,
               "svae_attn_bwd: workspace of %zu bytes is smaller than the required %zu", workspace_bytes,
               svae_attn_bwd_workspace_bytes(d));
  SVAE_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 256 == 0, SVAE_ERR_INVALID, "svae_attn_bwd: workspace must be 256-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (use_exact(d) || !sm100::bwd_supported(d)) return exact_bwd(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
  const bool ok = tma_ok(q, d->q_stride, d->heads, d->batch, d->seq_len) && tma_ok(k, d->k_stride, d->heads, d->batch, d->seq_len) &&
                  tma_ok(v, d->v_stride, d->heads, d->batch, d->seq_len) && tma_ok(out, d->o_stride, d->heads, d->batch, d->seq_len) &&
                  tma_ok(dout, d->do_stride, d->heads, d->batch, d->seq_len) && tma_ok(dq, d->dq_stride, d->heads, d->batch, d->seq_len) &&
                  tma_ok(dk, d->dk_stride, d->heads, d->batch, d->seq_len) && tma_ok(dv, d->dv_stride, d->heads, d->batch, d->seq_len);
  SVAE_REQUIRE(ok, SVAE_ERR_INVALID, "svae_attn_bwd: 16-bit tensors must be 16-byte aligned with strides that are multiples of 8 elements");
  if (use_one_pass(d)) return sm100::bwd1(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
  return sm100::bwd(d, q, k, v, out, dout, lse, kpm, dq, dk, dv, workspace, st);
}

