// Shared definitions of the sm_100a (tcgen05 / TMEM / TMA) attention kernels.
#pragma once

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace svae {
namespace sm100 {

constexpr int kTile = 128;        // rows of one MMA tile (queries in fwd / dQ, keys in dK/dV) = TMEM lanes
constexpr int kBlock = 32;        // SparseAttention.block_size
constexpr int kThreads = 160;     // warps 0-3: softmax / epilogue (one TMEM lane quarter each), warp 4: TMA + MMA issue
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
  static constexpr int fmt = 1;
  static constexpr CUtensorMapDataType tm = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __device__ static __forceinline__ float2 unpack(uint32_t u) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
  }
};
template <> struct Elem<__half> {
  static constexpr int fmt = 0;
  static constexpr CUtensorMapDataType tm = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __device__ static __forceinline__ float2 unpack(uint32_t u) { return __half22float2(*reinterpret_cast<__half2*>(&u)); }
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Byte offset of 16-byte chunk `chunk` of row `row` inside a TMA-swizzled tile whose rows are ROWB bytes
// (ROWB = 128 -> SWIZZLE_128B: chunk ^= row & 7;  ROWB = 64 -> SWIZZLE_64B: chunk ^= (row >> 1) & 3).
template <int ROWB>
__device__ __forceinline__ uint32_t swz_off(int row, int chunk) {
  if (ROWB == 128) return (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
  return (uint32_t)row * 64u + (uint32_t)((chunk ^ ((row >> 1) & 3)) << 4);
}

// Geometry of one 128-row tile against the banded + global-column layout.
//   fwd / dQ (query tile t):  slot 0 = key block 0 when cls; slots cls.. = key blocks lo .. lo+nband-1, lo = 4t-(left-1)
//   dK/dV   (key tile t):     slots 0..nband-1 = query blocks 4t-nsup .. ; (the global column is handled by the dQ pass)
struct TileGeom {
  int left, nsup, cls, causal;
  int nb;          // blocks in the sequence
  int nband;       // left + 3 + nsup
  int nslots;      // fwd/dQ: cls + nband ; dK/dV: nband
};

__host__ __device__ inline TileGeom make_geom(int window, int causal, int include_cls, int nb) {
  Band b = make_band(window, causal, include_cls);
  TileGeom g;
  g.left = b.left; g.nsup = b.nsup; g.cls = b.cls; g.causal = causal ? 1 : 0; g.nb = nb;
  g.nband = b.left + 3 + b.nsup;
  g.nslots = g.cls + g.nband;
  return g;
}

struct FwdParams {
  const float* kpm;     // [B, L] additive or null
  float* lse;           // [B, H, L]
  float* s_dump;        // debug: [B, H, L, nslots*32] raw scores, or null
  long long* timeline;  // debug: [num_ctas, 5 warps, 8] clock64 stamps, or null
  int L, H;
  TileGeom g;
  float scale_log2;     // scale * log2(e)
  int stagger_cycles;   // persistent kernel: delay of the second softmax group's first tile
};

struct BwdParams {
  const float* kpm;
  const float* lse;     // [B, H, L] natural log
  float* delta;         // [B, H, L] rowsum(dO * O): written by the dQ pass, read by the dK/dV pass
  float* gacc;          // [B, H, 2, 32, Dh] fp32: dK / dV of key block 0 (global column), atomically accumulated
  int L, H;
  TileGeom g;
  float scale, scale_log2;
  long long* timeline;  // debug: [2 kernels][num_ctas][3 roles (warp 0, warp 3, MMA warp)][16] clock64 stamps, or null
};

// ---- per-slot CUDA-core work on one row's 32 scores held in registers --------------------------------------
__device__ __forceinline__ void mask_above_diag(uint32_t (&v)[32], uint32_t below_diag) {
#pragma unroll
  for (int c = 0; c < 32; ++c)
    if (!((below_diag >> c) & 1u)) v[c] = 0xff800000u;      // -inf
}

// running max; fast path: raw scores (scaled once at the end), mask path: log2-domain with the additive mask
__device__ __forceinline__ float slot_max(const uint32_t (&v)[32], float m, bool has_kpm, const float* kp, float scale_log2) {
  if (!has_kpm) {
    float a = m, b = -INFINITY, c = -INFINITY, d = -INFINITY;
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
      a = ptx::fmax3(a, __uint_as_float(v[i + 0]), __uint_as_float(v[i + 1]));
      b = ptx::fmax3(b, __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
      c = ptx::fmax3(c, __uint_as_float(v[i + 4]), __uint_as_float(v[i + 5]));
      d = ptx::fmax3(d, __uint_as_float(v[i + 6]), __uint_as_float(v[i + 7]));
    }
    return ptx::fmax3(fmaxf(a, b), c, d);
  }
  float a0 = m, a1 = -INFINITY;
#pragma unroll
  for (int c = 0; c < 32; c += 2) {
    a0 = fmaxf(a0, fmaf(__uint_as_float(v[c]), scale_log2, kp[c]));
    a1 = fmaxf(a1, fmaf(__uint_as_float(v[c + 1]), scale_log2, kp[c + 1]));
  }
  return fmaxf(a0, a1);
}

// 2^x for two finite x <= 0 on the FMA pipe (no MUFU): Cody-Waite split by the 1.5 * 2^23 trick, degree-3 minimax
// polynomial of 2^f on [-0.5, 0.5] (relative error 7.5e-5, a sixth of an fp16 half-ulp), the integer part added into
// the exponent field.  Inputs below -125 are held there (2^-125: nothing for a row sum that contains a 1).
__device__ __forceinline__ float2 exp2_fma2(float2 x) {
  x = make_float2(fmaxf(x.x, -125.0f), fmaxf(x.y, -125.0f));
  const float2 r = fadd2(x, splat(12582912.0f));
  const float2 f = ffma2(fadd2(r, splat(-12582912.0f)), splat(-1.0f), x);
  float2 p = ffma2(splat(5.517165260e-02f), f, splat(2.426111209e-01f));
  p = ffma2(p, f, splat(6.932609885e-01f));
  p = ffma2(p, f, splat(9.999280737e-01f));
  return make_float2(__int_as_float((__float_as_int(r.x) << 23) + __float_as_int(p.x)),
                     __int_as_float((__float_as_int(r.y) << 23) + __float_as_int(p.y)));
}

// Without a padding mask every second pair of exponentials is evaluated on the FMA pipe (exp2_fma2) instead of MUFU.EX2:
// the exp pass is MUFU-bound (8.2 cycles per warp instruction and SMSP) while the FMA pipe idles.  Causally masked
// scores (-inf) come out as 2^-125 there instead of 0 -- nothing against a row sum that holds the row's own diagonal
// key; rows without any finite key only exist with a padding mask, which takes the MUFU-only path below.
template <typename T>
__device__ __forceinline__ void slot_exp_pack(const uint32_t (&v)[32], uint32_t (&pk)[16], float& l0, float& l1, bool has_kpm,
                                              const float* kp, float scale_log2, float neg_m) {
  if (!has_kpm) {
    float2 l = make_float2(l0, l1);
#pragma unroll
    for (int c = 0; c < 32; c += 2) {
      const float2 x = ffma2(make_float2(__uint_as_float(v[c]), __uint_as_float(v[c + 1])), splat(scale_log2), splat(neg_m));
      const float2 pe = ((c >> 1) & 1) ? exp2_fma2(x) : make_float2(fast_exp2(x.x), fast_exp2(x.y));
      l = fadd2(l, pe);
      pk[c >> 1] = Elem<T>::pack(pe.x, pe.y);
    }
    l0 = l.x;
    l1 = l.y;
  } else {
#pragma unroll
    for (int c = 0; c < 32; c += 2) {
      const float p0 = fast_exp2(fmaf(__uint_as_float(v[c]), scale_log2, kp[c]) + neg_m);
      const float p1 = fast_exp2(fmaf(__uint_as_float(v[c + 1]), scale_log2, kp[c + 1]) + neg_m);
      l0 += p0;
      l1 += p1;
      pk[c >> 1] = Elem<T>::pack(p0, p1);
    }
  }
}


int encode_tmap(CUtensorMap* map, CUtensorMapDataType dt, const void* base, int Dh, int L, int H, int B,
                const int64_t stride[3], int box_rows);
// 2-D map over a row-major 16-bit [rows, cols] matrix (row stride ld elements); box = 64 columns (one SWIZZLE_128B
// row) x box_rows rows.  Rows past the end read as zeros.
int encode_tmap_2d(CUtensorMap* map, CUtensorMapDataType dt, const void* base, int64_t cols, int64_t rows, int64_t ld,
                   int box_rows);

}  // namespace sm100
}  // namespace svae
