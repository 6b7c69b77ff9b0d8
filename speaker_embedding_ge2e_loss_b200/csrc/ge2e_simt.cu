// SIMT fp32 path of the GE2E loss (exact-parity path, any N / M >= 2 / D <= 1024).
//
// Kernels
//   prep_kernel      one CTA per speaker: L2-normalise, centroid, leave-one-out cosine
//                    (reference s3:33-38, s3:95-112, s3:57)
//   strip_kernel     the similarity contraction fused with its consumer.  Each warp owns R
//                    "owner" rows in registers (lanes split D, 128-bit loads); "stream" rows
//                    pass through shared memory 32 at a time.  Dot products are reduced with a
//                    transposing warp-shuffle butterfly so that lane l ends up holding the dot
//                    product against stream row l; the softmax / contrast epilogue then runs
//                    one column per lane.  Three modes:
//                      FWD     owner = utterances, stream = centroids -> online LSE / argmax
//                      BWD_DE  owner = utterances, stream = centroids -> dE_hat = (wG) C_hat
//                      BWD_DC  owner = centroids,  stream = utterances -> dC_hat = (wG)^T E_hat
//                    (reference s3:64-79, s3:27, s3:114-127 and their autograd)
//   contrast_bwd     the contrast gradient has two non-zeros per row: gather/scatter kernel
//   finalize_kernel  one CTA per speaker: diagonal term, normalisation Jacobians, fan-out
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <limits.h>

#include <algorithm>
#include <stdlib.h>

#include <initializer_list>
#include <type_traits>

#include "ge2e_common.cuh"
#include "ge2e_tc_ptx.cuh"

namespace ge2e {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / kWarp;
constexpr int kStreamRows = 32;  // stream rows per shared-memory stage (= warp width)

enum { MODE_FWD = 0, MODE_BWD_DE = 1, MODE_BWD_DC = 2 };

__device__ __forceinline__ float4 ld4(const float* __restrict__ row, int col, int D, bool vec) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (vec) {
    if (col < D) v = __ldg(reinterpret_cast<const float4*>(row + col));
  } else {
    if (col + 0 < D) v.x = __ldg(row + col + 0);
    if (col + 1 < D) v.y = __ldg(row + col + 1);
    if (col + 2 < D) v.z = __ldg(row + col + 2);
    if (col + 3 < D) v.w = __ldg(row + col + 3);
  }
  return v;
}

// same without the read-only path: for data written earlier in the same kernel
__device__ __forceinline__ float4 ld4_plain(const float* row, int col, int D, bool vec) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (vec) {
    if (col < D) v = *reinterpret_cast<const float4*>(row + col);
  } else {
    if (col + 0 < D) v.x = row[col + 0];
    if (col + 1 < D) v.y = row[col + 1];
    if (col + 2 < D) v.z = row[col + 2];
    if (col + 3 < D) v.w = row[col + 3];
  }
  return v;
}

__device__ __forceinline__ void st4(float* __restrict__ row, int col, int D, bool vec, float4 v) {
  if (vec) {
    if (col < D) *reinterpret_cast<float4*>(row + col) = v;
  } else {
    if (col + 0 < D) row[col + 0] = v.x;
    if (col + 1 < D) row[col + 1] = v.y;
    if (col + 2 < D) row[col + 2] = v.z;
    if (col + 3 < D) row[col + 3] = v.w;
  }
}

__device__ __forceinline__ float dot4(float4 a, float4 b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}

// Physical row of logical row r.  The optional row index folds the trainer's `embeddings[unperm]`
// gather (s4_train_embed_model.py:189-192) into the loads of prep / finalize and the scatter of its
// backward into finalize's stores; nullptr = rows are already in [speaker][utterance] order.
__device__ __forceinline__ size_t phys_row(const int32_t* __restrict__ idx, size_t r) {
  return idx != nullptr ? static_cast<size_t>(__ldg(idx + r)) : r;
}

// four consecutive elements of T at an aligned address: 16 bytes for fp32, 8 bytes for the half types
template <typename T>
__device__ __forceinline__ bool is_vec(const T* p, int D) {
  return ((D & 3) == 0) && ((reinterpret_cast<uintptr_t>(p) & (4 * sizeof(T) - 1)) == 0);
}

// ---- element types of E and dE (ge2e_dtype) ---------------------------------------------------
// E is fp32, bf16 or fp16; a half-type element is widened to fp32 when it is loaded, and every number after that
// load is the fp32 path's.  dE is fp32 or E's type; it is rounded to its type (nearest even) once, when it is
// stored.  Everything between prep and finalize (e_hat, c_hat, the row statistics, dE_hat, dC_hat) stays fp32.
__device__ __forceinline__ float to_f(__half x) { return __half2float(x); }
__device__ __forceinline__ float to_f(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f(float x);
template <> __device__ __forceinline__ float from_f<float>(float x) { return x; }
template <> __device__ __forceinline__ __half from_f<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// four half-type elements (8 bytes) <-> a float4
template <typename T> __device__ __forceinline__ float4 widen4(uint2 r);
template <> __device__ __forceinline__ float4 widen4<__nv_bfloat16>(uint2 r) {
  return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                     __uint_as_float(r.y & 0xffff0000u));
}
template <> __device__ __forceinline__ float4 widen4<__half>(uint2 r) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
template <typename T> __device__ __forceinline__ uint2 narrow4(float4 v);
template <> __device__ __forceinline__ uint2 narrow4<__nv_bfloat16>(float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}
template <> __device__ __forceinline__ uint2 narrow4<__half>(float4 v) {
  const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}

// four elements of T as one vector: a float4 for fp32, 8 bytes for the half types
template <typename T>
using vec4_t = typename std::conditional<std::is_same<T, float>::value, float4, uint2>::type;
template <typename T>
__device__ __forceinline__ float4 ldg4v(const vec4_t<T>* p) {     // read-only path
  if constexpr (std::is_same<T, float>::value) return __ldg(p);
  else return widen4<T>(__ldg(p));
}
template <typename T>
__device__ __forceinline__ void st4vv(vec4_t<T>* p, float4 v) {
  if constexpr (std::is_same<T, float>::value) *p = v;
  else *p = narrow4<T>(v);
}
// elements [0, 4) at p (is_vec-aligned)
template <typename T>
__device__ __forceinline__ float4 ldg4(const T* p) { return ldg4v<T>(reinterpret_cast<const vec4_t<T>*>(p)); }
template <typename T>
__device__ __forceinline__ void st4v(T* p, float4 v) { st4vv<T>(reinterpret_cast<vec4_t<T>*>(p), v); }
// ld4 / st4 for any element type (tail-safe; vec = is_vec of the row base)
template <typename T>
__device__ __forceinline__ float4 ld4e(const T* __restrict__ row, int col, int D, bool vec) {
  if constexpr (std::is_same<T, float>::value) {
    return ld4(row, col, D, vec);
  } else {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec) {
      if (col < D) v = ldg4(row + col);
    } else {
      if (col + 0 < D) v.x = to_f(__ldg(row + col + 0));
      if (col + 1 < D) v.y = to_f(__ldg(row + col + 1));
      if (col + 2 < D) v.z = to_f(__ldg(row + col + 2));
      if (col + 3 < D) v.w = to_f(__ldg(row + col + 3));
    }
    return v;
  }
}
template <typename T>
__device__ __forceinline__ void st4e(T* __restrict__ row, int col, int D, bool vec, float4 v) {
  if constexpr (std::is_same<T, float>::value) {
    st4(row, col, D, vec, v);
  } else {
    if (vec) {
      if (col < D) st4v(row + col, v);
    } else {
      if (col + 0 < D) row[col + 0] = from_f<T>(v.x);
      if (col + 1 < D) row[col + 1] = from_f<T>(v.y);
      if (col + 2 < D) row[col + 2] = from_f<T>(v.z);
      if (col + 3 < D) row[col + 3] = from_f<T>(v.w);
    }
  }
}

// ------------------------------------------------------------------------------------------
// Row arithmetic of prep and finalize, shared by every body (generic, warp, register, single-kernel step).
// Speaker j has rows e_i, column sum s = sum_i e_i, centroid c = s / M (s3:37) and leave-one-out centroids
// u_i = d_i / (M - 1) with d_i = s - e_i (s3:105-111).  The bodies reduce the raw sums |e|^2, |d|^2, e.d, |s|^2,
// e.dE_hat and s.dC_hat however their threads map to rows and columns; the helpers below take those sums.
// ------------------------------------------------------------------------------------------
struct RowNorms {
  float ne, nu;           // |e|, |u|
  float inv_ne, inv_nu;   // 1 / max(|e|, delta), 1 / max(|u|, delta)
  float cos;              // e_hat . u_hat (s3:57)
};
__device__ __forceinline__ RowNorms row_norms(float ne2, float nd2, float ed, float inv_m1) {
  RowNorms n;
  n.ne = sqrtf(ne2);
  n.nu = sqrtf(nd2) * inv_m1;
  n.inv_ne = 1.f / fmaxf(n.ne, kCosDelta);
  n.inv_nu = 1.f / fmaxf(n.nu, kCosDelta);
  n.cos = (ed * inv_m1) * n.inv_ne * n.inv_nu;
  return n;
}

// c_hat = s * centroid_scale(|s|^2, 1 / M)
__device__ __forceinline__ float centroid_scale(float ss, float inv_m) {
  return inv_m / fmaxf(sqrtf(ss) * inv_m, kCosDelta);
}

// dd = w G_jj, the diagonal element of w G of a row with upstream gradient g_r.  aux is the row's row_aux for
// softmax (q = 1 - p_jj: G_jj = g_r (p_jj - 1)) and its cos_diag for contrast (G_jj = -g_r sigma'(S_jj)).
__device__ __forceinline__ float diag_term(int variant, float g_r, float aux, float w, float b, float eps) {
  float Gd;
  if (variant == GE2E_SOFTMAX) {
    Gd = -g_r * aux;
  } else {
    const float sp = 1.f / (1.f + expf(-fmaf(w, aux + eps, b)));
    Gd = -g_r * sp * (1.f - sp);
  }
  return w * Gd;
}

// Gradient of one row through e_hat and u_hat.  The row's gradients are d e_hat = gsc dE_hat + dd u_hat and
// d u_hat = dd e_hat (its diagonal cosine); through the two normalisations (clamp_proj_scale)
//   de = (d e_hat - e_hat (e_hat . d e_hat) s_e) inv_ne,   du = (d u_hat - u_hat (u_hat . d u_hat) s_u) inv_nu.
// With e_hat = e inv_ne and u_hat = d inv_nu / (M - 1) both are linear in dE_hat, e and d:
//   de = a_g dE_hat + a_e e + a_d d,   du = b_e e + b_d d.
// gsc: factor of un-normalised dE_hat rows (else 1); eg = (e . dE_hat) gsc.
struct RowJacobian {
  float a_g, a_e, a_d, b_e, b_d;
  __device__ __forceinline__ float de(float e, float d, float g) const { return a_g * g + a_e * e + a_d * d; }
  __device__ __forceinline__ float du(float e, float d) const { return b_e * e + b_d * d; }
};
__device__ __forceinline__ RowJacobian row_jacobian(const RowNorms& n, float eg, float gsc, float dd, float inv_m1) {
  float proj_e = eg * n.inv_ne + dd * n.cos;   // e_hat . d e_hat
  float proj_u = dd * n.cos;                   // u_hat . d u_hat
  if (n.ne < kCosDelta) proj_e *= clamp_proj_scale(n.ne);
  if (n.nu < kCosDelta) proj_u *= clamp_proj_scale(n.nu);
  RowJacobian J;
  J.a_g = n.inv_ne * gsc;
  J.a_e = -proj_e * n.inv_ne * n.inv_ne;
  J.a_d = dd * n.inv_nu * inv_m1 * n.inv_ne;
  J.b_e = dd * n.inv_ne * n.inv_nu;
  J.b_d = -proj_u * n.inv_nu * n.inv_nu * inv_m1;
  return J;
}

// Gradient of the centroid through c_hat = s inv / M (clamp_proj_scale), divided by M for the fan-out to the rows:
//   dc / M = (dC_hat - c_hat (c_hat . dC_hat) s_c) inv / M = k.x dC_hat - k.y s,   sdc = s . dC_hat
__device__ __forceinline__ float2 centroid_jacobian(float ss, float sdc, float inv_m) {
  const float nc = sqrtf(ss) * inv_m;
  const float inv = 1.f / fmaxf(nc, kCosDelta);
  float proj = (sdc * inv_m) * inv;            // c_hat . dC_hat
  if (nc < kCosDelta) proj *= clamp_proj_scale(nc);
  return make_float2(inv * inv_m, proj * inv * inv * inv_m * inv_m);
}

// ------------------------------------------------------------------------------------------
// K1: prep.  grid = n_local, block = 256, dynamic smem = (M + 1) * Dp floats.
// ------------------------------------------------------------------------------------------
// The M raw rows of speaker j, widened to fp32, into sE[M][Dp] (columns D..Dp-1 zero); ends with a __syncthreads.
template <typename TE>
__device__ __forceinline__ void stage_rows(const TE* __restrict__ E, const int32_t* __restrict__ idx, int j, int M,
                                           int D, int Dp, float* sE) {
  const bool vec_in = is_vec(E, D);
  for (int v = threadIdx.x; v < M * (Dp >> 2); v += kThreads) {
    const int i = v / (Dp >> 2), col = (v % (Dp >> 2)) << 2;
    *reinterpret_cast<float4*>(&sE[(size_t)i * Dp + col]) =
        ld4e(E + phys_row(idx, (size_t)j * M + i) * D, col, D, vec_in);
  }
  __syncthreads();
}

// Body shared by prep_kernel and the fused small-batch kernel: speaker j, block of kThreads threads,
// `smem` = (M + 1) * Dp floats.
template <bool ROUND, typename TE = float>
__device__ __forceinline__ void prep_body(const TE* __restrict__ E, const int32_t* __restrict__ idx, int j, int M,
                                          int D, int Dp, float* __restrict__ e_hat, float* __restrict__ c_hat,
                                          float* __restrict__ cos_diag, float* smem) {
  __shared__ float red[kWarps];
  __shared__ float s_sc;
  float* sE = smem;                    // [M][Dp]
  float* sS = smem + (size_t)M * Dp;   // [Dp] column sums
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const bool vec_out = is_vec(e_hat, D);

  stage_rows(E, idx, j, M, D, Dp, sE);
  for (int d = tid; d < Dp; d += kThreads) {
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += sE[(size_t)i * Dp + d];   // s3:105
    sS[d] = s;
  }
  __syncthreads();

  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  for (int i = wid; i < M; i += kWarps) {
    float ne2 = 0.f, nd2 = 0.f, ed = 0.f;
    for (int d = lane << 2; d < Dp; d += 128) {
      const float4 e = *reinterpret_cast<const float4*>(&sE[(size_t)i * Dp + d]);
      const float4 s = *reinterpret_cast<const float4*>(&sS[d]);
      const float4 dv = make_float4(s.x - e.x, s.y - e.y, s.z - e.z, s.w - e.w);
      ne2 += dot4(e, e); nd2 += dot4(dv, dv); ed += dot4(e, dv);
    }
    const RowNorms n = row_norms(warp_sum(ne2), warp_sum(nd2), warp_sum(ed), inv_m1);
    float* out = e_hat + ((size_t)j * M + i) * D;
    for (int d = lane << 2; d < Dp; d += 128) {
      float4 e = *reinterpret_cast<const float4*>(&sE[(size_t)i * Dp + d]);
      e.x *= n.inv_ne; e.y *= n.inv_ne; e.z *= n.inv_ne; e.w *= n.inv_ne;
      if (ROUND) { e.x = round_tf32(e.x); e.y = round_tf32(e.y); e.z = round_tf32(e.z); e.w = round_tf32(e.w); }
      st4(out, d, D, vec_out, e);
    }
    if (lane == 0) cos_diag[(size_t)j * M + i] = n.cos;
  }

  float part = 0.f;
  for (int d = tid; d < Dp; d += kThreads) part += sS[d] * sS[d];
  const float tot = block_sum(part, red);
  if (tid == 0) s_sc = centroid_scale(tot, inv_m);
  __syncthreads();
  const float sc = s_sc;
  for (int d = tid; d < D; d += kThreads) {
    float c = sS[d] * sc;
    if (ROUND) c = round_tf32(c);
    c_hat[(size_t)j * D + d] = c;
  }
}

template <bool ROUND, typename TE>
__global__ void __launch_bounds__(kThreads)
prep_kernel(const TE* __restrict__ E, const int32_t* __restrict__ idx, int M, int D, int Dp,
            float* __restrict__ e_hat, float* __restrict__ c_hat, float* __restrict__ cos_diag,
            float* __restrict__ accum) {
  extern __shared__ __align__(16) float smem[];
  if (blockIdx.x == 0 && threadIdx.x < 4 && accum != nullptr) accum[threadIdx.x] = 0.f;
  prep_body<ROUND>(E, idx, blockIdx.x, M, D, Dp, e_hat, c_hat, cos_diag, smem);
}


// ------------------------------------------------------------------------------------------
// K1 (fast path): one WARP per speaker, no shared memory, no block barriers, no divisions.
// Lane l owns the float4 columns {4 l + 128 c}.  Pass 1 sums the speaker's rows (s3:105), pass 2
// re-reads them (L1 hits) for the norms / leave-one-out cosine (s3:57) and writes e_hat.
// Requires D = 128 KCH, 16-byte aligned rows.  grid = ceil(n_local / 4), block = 128.
// ------------------------------------------------------------------------------------------
// Operand precision of the normalised rows (PREC): 0 = fp32 as they are, 1 = rounded to TF32, 2 = two fp16 planes
// hi = fp16(x), lo = fp16(x - hi), laid out [rows][2][D] -- a row's hi plane then its lo plane in the bytes of the
// fp32 row, so whatever moves rows (all-gather, peer publish) moves both planes (the tensor-core path's fp32-class
// mode: hi.hi + hi.lo + lo.hi reproduces the fp32 product to ~2^-22).  put4 stores columns [col, col + 4) of `row`.
template <int PREC>
__device__ __forceinline__ void put4(float* base, size_t row, int D, int col, float4 v) {
  if (PREC == 3) {          // the hi plane alone (fp16 operands of the TF32-tolerance class)
    __half* h = reinterpret_cast<__half*>(base);
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    uint2 hi;
    hi.x = *reinterpret_cast<const uint32_t*>(&h0); hi.y = *reinterpret_cast<const uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(h + row * 2 * D + col) = hi;
  } else if (PREC == 2) {
    __half* h = reinterpret_cast<__half*>(base);
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    const __half2 l0 = __floats2half2_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2half2_rn(v.z - f1.x, v.w - f1.y);
    uint2 hi, lo;
    hi.x = *reinterpret_cast<const uint32_t*>(&h0); hi.y = *reinterpret_cast<const uint32_t*>(&h1);
    lo.x = *reinterpret_cast<const uint32_t*>(&l0); lo.y = *reinterpret_cast<const uint32_t*>(&l1);
    *reinterpret_cast<uint2*>(h + row * 2 * D + col) = hi;
    *reinterpret_cast<uint2*>(h + row * 2 * D + D + col) = lo;
  } else {
    if (PREC == 1) { v.x = round_tf32(v.x); v.y = round_tf32(v.y); v.z = round_tf32(v.z); v.w = round_tf32(v.w); }
    *reinterpret_cast<float4*>(base + row * D + col) = v;
  }
}

constexpr int kPrepWarps = 4;
constexpr int kRowBatch = 4;   // rows in flight per lane (KCH float4 loads each)
constexpr int kRegRows = 16;   // register-resident variants hold up to this many rows per speaker
constexpr int kRegBlocksPerSM = 4;   // register-resident variants: <= 128 registers, 16 warps resident per SM

template <int KCH, int PREC, typename TE>
__global__ void __launch_bounds__(kPrepWarps * 32)
prep_warp_kernel(const TE* __restrict__ E, const int32_t* __restrict__ idx, int n_local, int M,
                 float* __restrict__ e_hat, float* __restrict__ c_hat, float* __restrict__ cos_diag,
                 float* __restrict__ accum) {
  constexpr int D = KCH * 128;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int j = blockIdx.x * kPrepWarps + wid;
  pdl_wait();        // before touching memory: the previous step's kernels may still read what this one writes
  pdl_trigger();     // the forward tensor-core kernel may set itself up while this grid runs
  if (blockIdx.x == 0 && threadIdx.x < 4 && accum != nullptr) accum[threadIdx.x] = 0.f;
  if (j >= n_local) return;
  auto rowp = [&](int i) {      // + c * 32 vectors per 128-column chunk
    return reinterpret_cast<const vec4_t<TE>*>(E + phys_row(idx, (size_t)j * M + i) * D) + lane;
  };
  float4 s[KCH];
#pragma unroll
  for (int c = 0; c < KCH; ++c) s[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i0 = 0; i0 < M; i0 += kRowBatch) {
    float4 v[kRowBatch][KCH];
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r)
#pragma unroll
      for (int c = 0; c < KCH; ++c)
        v[r][c] = (i0 + r < M) ? ldg4v<TE>(rowp(i0 + r) + c * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r)
#pragma unroll
      for (int c = 0; c < KCH; ++c) {
        s[c].x += v[r][c].x; s[c].y += v[r][c].y; s[c].z += v[r][c].z; s[c].w += v[r][c].w;
      }
  }
  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  float ss = 0.f;
#pragma unroll
  for (int c = 0; c < KCH; ++c) ss += dot4(s[c], s[c]);
  const float sc = centroid_scale(warp_sum(ss), inv_m);
#pragma unroll
  for (int c = 0; c < KCH; ++c)
    put4<PREC>(c_hat, j, D, 4 * lane + 128 * c,
               make_float4(s[c].x * sc, s[c].y * sc, s[c].z * sc, s[c].w * sc));
  float my_cos = 0.f;
  for (int i0 = 0; i0 < M; i0 += kRowBatch) {
    float4 v[kRowBatch][KCH];
    float ne2[kRowBatch], nd2[kRowBatch], ed[kRowBatch];
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r)
#pragma unroll
      for (int c = 0; c < KCH; ++c)
        v[r][c] = (i0 + r < M) ? ldg4v<TE>(rowp(i0 + r) + c * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r) {
      ne2[r] = 0.f; nd2[r] = 0.f; ed[r] = 0.f;
#pragma unroll
      for (int c = 0; c < KCH; ++c) {
        const float4 e = v[r][c];
        const float4 d = make_float4(s[c].x - e.x, s[c].y - e.y, s[c].z - e.z, s[c].w - e.w);
        ne2[r] += dot4(e, e); nd2[r] += dot4(d, d); ed[r] += dot4(e, d);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < kRowBatch; ++r) {
        ne2[r] += __shfl_xor_sync(0xffffffffu, ne2[r], o);
        nd2[r] += __shfl_xor_sync(0xffffffffu, nd2[r], o);
        ed[r] += __shfl_xor_sync(0xffffffffu, ed[r], o);
      }
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r) {
      if (i0 + r < M) {
        const RowNorms n = row_norms(ne2[r], nd2[r], ed[r], inv_m1);
        if (lane == ((i0 + r) & 31)) my_cos = n.cos;
#pragma unroll
        for (int c = 0; c < KCH; ++c) {
          float4 e = v[r][c];
          e.x *= n.inv_ne; e.y *= n.inv_ne; e.z *= n.inv_ne; e.w *= n.inv_ne;
          put4<PREC>(e_hat, (size_t)j * M + i0 + r, D, 4 * lane + 128 * c, e);
        }
      }
    }
    // flush the cosines every 32 rows (one coalesced store per 32 rows)
    if (((i0 + kRowBatch) & 31) == 0 || i0 + kRowBatch >= M) {
      const int base = (i0 + kRowBatch - 1) & ~31;
      if (base + lane < M) cos_diag[(size_t)j * M + base + lane] = my_cos;
    }
  }
}

// ------------------------------------------------------------------------------------------
// K1 (register-resident variant, M <= 16, D = 128 W): W warps per speaker, warp w of the speaker
// owning the columns [128 w, 128 w + 128), so a lane holds one float4 of every row.  Every row is
// loaded ONCE, all loads in flight together, and kept in registers.  The per-row sums go through a
// transposing butterfly (reduce16_transposed): lane l ends up with the warp's partial of row
// rev4(l & 15); the W partials are added through shared memory (speaker_sum), so the square roots
// / reciprocals of all rows are evaluated once, lane-parallel, instead of row after row.  At cfg3
// there are a few warps per scheduler and the kernel time is the latency of one warp's dependency
// chain; splitting the columns over W warps halves that chain's loads and arithmetic at D = 256.
// ------------------------------------------------------------------------------------------
__host__ __device__ constexpr int rev4(int i) {
  return ((i & 1) << 3) | ((i & 2) << 1) | ((i & 4) >> 1) | ((i & 8) >> 3);
}
// warp total of v[rev4(lane & 15)]: 16 shuffles for 16 values
__device__ __forceinline__ float reduce16_transposed(const float (&v)[16], int lane) {
  float a[8], b[4], c[2];
  const bool u1 = (lane & 1) != 0, u2 = (lane & 2) != 0, u4 = (lane & 4) != 0, u8 = (lane & 8) != 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) a[q] = (u1 ? v[q + 8] : v[q]) + __shfl_xor_sync(0xffffffffu, u1 ? v[q] : v[q + 8], 1);
#pragma unroll
  for (int q = 0; q < 4; ++q) b[q] = (u2 ? a[q + 4] : a[q]) + __shfl_xor_sync(0xffffffffu, u2 ? a[q] : a[q + 4], 2);
#pragma unroll
  for (int q = 0; q < 2; ++q) c[q] = (u4 ? b[q + 2] : b[q]) + __shfl_xor_sync(0xffffffffu, u4 ? b[q] : b[q + 2], 4);
  const float e = (u8 ? c[1] : c[0]) + __shfl_xor_sync(0xffffffffu, u8 ? c[0] : c[1], 8);
  return e + __shfl_xor_sync(0xffffffffu, e, 16);
}

// Speaker totals of Q quantities from the partials of the speaker's W warps (warps W s ... W s + W - 1 of the
// block).  Lane l's x[q] is either a per-row partial of row rev4(l & 15) (reduce16_transposed) or a per-speaker
// scalar (the same in every lane); either way lanes l and l + 16 agree, so 16 slots per quantity carry it.  The
// partials are added in warp order: every warp of the speaker gets the same bits.  One named barrier per speaker,
// so a speaker whose warps returned early holds up nobody.  W = 1 is a no-op.
template <int W, int Q>
__device__ __forceinline__ void speaker_sum(float (&x)[Q], float (*xch)[Q][16], int wid, int lane) {
  if (W == 1) return;
  if (lane < 16) {
#pragma unroll
    for (int q = 0; q < Q; ++q) xch[wid][q][lane] = x[q];
  }
  asm volatile("bar.sync %0, %1;" ::"r"(1 + wid / W), "r"(W * 32) : "memory");
  const int first = wid - wid % W;
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    float t = xch[first][q][lane & 15];
#pragma unroll
    for (int w = 1; w < W; ++w) t += xch[first + w][q][lane & 15];
    x[q] = t;
  }
}

template <int W, int RR, int PREC, typename TE>
__global__ void __launch_bounds__(kPrepWarps * 32, kRegBlocksPerSM)
prep_reg_kernel(const TE* __restrict__ E, const int32_t* __restrict__ idx, int n_local, int M,
                float* __restrict__ e_hat, float* __restrict__ c_hat, float* __restrict__ cos_diag,
                float* __restrict__ accum) {
  constexpr int D = W * 128, R = RR;       // rows held in registers (M <= R <= 16)
  static_assert(R <= 16, "reduce16_transposed handles 16 rows");
  static_assert(kPrepWarps % W == 0, "a block holds whole speakers");
  __shared__ float xch[kPrepWarps][4][16];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int j = blockIdx.x * (kPrepWarps / W) + wid / W;
  const int col = 128 * (wid % W) + 4 * lane;     // this lane's four columns of every row
  pdl_wait();        // before touching memory: the previous step's kernels may still read what this one writes
  pdl_trigger();     // the forward tensor-core kernel may set itself up while this grid runs
  if (blockIdx.x == 0 && threadIdx.x < 4 && accum != nullptr) accum[threadIdx.x] = 0.f;
  if (j >= n_local) return;     // all W warps of the speaker
  float4 v[R];
#pragma unroll
  for (int i = 0; i < R; ++i)
    v[i] = (i < M) ? ldg4(E + phys_row(idx, (size_t)j * M + i) * D + col) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 s = v[0];
#pragma unroll
  for (int i = 1; i < R; ++i) { s.x += v[i].x; s.y += v[i].y; s.z += v[i].z; s.w += v[i].w; }
  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  float ne2[16], nd2[16], ed[16];
#pragma unroll
  for (int i = R; i < 16; ++i) { ne2[i] = 0.f; nd2[i] = 0.f; ed[i] = 0.f; }
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const float4 e = v[i];
    const float4 d = make_float4(s.x - e.x, s.y - e.y, s.z - e.z, s.w - e.w);
    ne2[i] = dot4(e, e); nd2[i] = dot4(d, d); ed[i] = dot4(e, d);
  }
  float t[4] = {reduce16_transposed(ne2, lane), reduce16_transposed(nd2, lane), reduce16_transposed(ed, lane),
                warp_sum(dot4(s, s))};
  speaker_sum<W>(t, xch, wid, lane);
  const float sc = centroid_scale(t[3], inv_m);
  put4<PREC>(c_hat, j, D, col, make_float4(s.x * sc, s.y * sc, s.z * sc, s.w * sc));
  const int my_row = rev4(lane & 15);
  const float inv_ne = row_norms(t[0], t[1], t[2], inv_m1).inv_ne;
  if (wid % W == 0 && lane < 16 && my_row < M)     // the cosine in the storing lanes only
    cos_diag[(size_t)j * M + my_row] = row_norms(t[0], t[1], t[2], inv_m1).cos;
#pragma unroll
  for (int i = 0; i < R; ++i) {
    if (i < M) {      // warp-uniform
      const float k = __shfl_sync(0xffffffffu, inv_ne, rev4(i));
      float4 e = v[i];
      e.x *= k; e.y *= k; e.z *= k; e.w *= k;
      put4<PREC>(e_hat, (size_t)j * M + i, D, col, e);
    }
  }
}

// ------------------------------------------------------------------------------------------
// strip kernel
// ------------------------------------------------------------------------------------------
struct StripParams {
  const float* own;   // [n_own, D]
  const float* str;   // [n_str, D]
  int n_own, n_str, D;
  int M, spk_offset;  // local utterance row r belongs to global speaker spk_offset + r / M
  const float* cos_diag;
  const float* row_stat;   // bwd: lse per local utterance row
  const float* row_aux;    // bwd: q = 1 - p_jj per local utterance row
  float* row_aux_out;      // fwd softmax
  const float* w;
  const float* b;
  const float* grad_out;
  const float* grad_rows;  // bwd, RG instantiations: upstream gradient per local utterance row (replaces grad_out)
  float eps;
  float* row_stat_out;     // fwd
  int32_t* kstar_out;      // fwd contrast
  float* loss_accum;       // fwd
  float* per_row_out;      // fwd optional
  float* sim_out;          // fwd optional [n_own, n_str]
  float* acc_out;          // bwd: dE_hat [n_own, D] or dC_hat_partial [n_own, D]
  float* dwdb;             // bwd_de
  int chunks_per_split;    // stream chunks handled per blockIdx.y
};

// Transposing butterfly: after RedT<0>::run, lane l holds (for each owner row q) the full dot
// product against stream row t0 + l.  31 shuffles per owner row instead of 32 x 5.
template <int K, int R, int KCH>
struct RedT {
  static __device__ __forceinline__ void run(const float4 (&a)[R][KCH], const float* __restrict__ stage,
                                             int t, int lane, float (&out)[R]) {
    float lo[R], hi[R];
    RedT<K + 1, R, KCH>::run(a, stage, t, lane, lo);
    RedT<K + 1, R, KCH>::run(a, stage, t + (1 << K), lane, hi);
    const bool up = (lane & (1 << K)) != 0;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const float send = up ? lo[q] : hi[q];
      const float keep = up ? hi[q] : lo[q];
      out[q] = keep + __shfl_xor_sync(0xffffffffu, send, 1 << K);
    }
  }
};
template <int R, int KCH>
struct RedT<5, R, KCH> {
  static __device__ __forceinline__ void run(const float4 (&a)[R][KCH], const float* __restrict__ stage,
                                             int t, int lane, float (&out)[R]) {
#pragma unroll
    for (int q = 0; q < R; ++q) out[q] = 0.f;
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      const float4 bv = *reinterpret_cast<const float4*>(&stage[(size_t)t * (KCH * 128) + c * 128 + (lane << 2)]);
#pragma unroll
      for (int q = 0; q < R; ++q) out[q] += dot4(a[q][c], bv);
    }
  }
};

// RG: the upstream gradient is one value per utterance row (p.grad_rows) instead of the scalar p.grad_out
template <int MODE, int VARIANT, int KCH, int R, bool RG = false>
__global__ void __launch_bounds__(kThreads)
strip_kernel(const StripParams p) {
  extern __shared__ __align__(16) float stage[];   // [32][KCH*128]
  __shared__ float red[kWarps];
  constexpr int ROWLEN = KCH * 128;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int own0 = (blockIdx.x * kWarps + wid) * R;
  const int D = p.D;
  const bool vec_own = is_vec(p.own, D), vec_str = is_vec(p.str, D);
  const float w = __ldg(p.w), b = __ldg(p.b), eps = p.eps;
  const float g = (MODE == MODE_FWD || RG) ? 1.f : __ldg(p.grad_out);

  float4 a[R][KCH];
#pragma unroll
  for (int q = 0; q < R; ++q) {
    const int row = own0 + q;
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      const int col = (lane << 2) + c * 128;
      a[q][c] = (row < p.n_own) ? ld4(p.own + (size_t)row * D, col, D, vec_own) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }

  // per-owner-row state
  int jg[R];        // FWD / BWD_DE: global speaker of the owner utterance row
  float cd[R];      // cos_diag of the owner row
  float lse[R];     // BWD_DE
  float qd[R];      // BWD_DE: 1 - p_jj
  float gr[R];      // BWD_DE: upstream gradient of the owner row
  float m_run[R], l_run[R];   // FWD softmax (per lane, merged at the end)
  float best[R]; int bestk[R];  // FWD contrast
  float4 acc[R][KCH];
  float dw_acc = 0.f;
#pragma unroll
  for (int q = 0; q < R; ++q) {
    const int row = own0 + q;
    // rows past the end: lse = +inf makes every G of that row exactly 0
    jg[q] = -1; cd[q] = 0.f; lse[q] = INFINITY; qd[q] = 0.f; gr[q] = g;
    if (MODE != MODE_BWD_DC && row < p.n_own) {
      jg[q] = p.spk_offset + row / p.M;
      cd[q] = __ldg(p.cos_diag + row);
      if (MODE == MODE_BWD_DE) { lse[q] = __ldg(p.row_stat + row); qd[q] = __ldg(p.row_aux + row); }
      if (MODE == MODE_BWD_DE && RG) gr[q] = __ldg(p.grad_rows + row);
    }
    m_run[q] = -INFINITY; l_run[q] = 0.f; best[q] = -INFINITY; bestk[q] = INT_MAX;
#pragma unroll
    for (int c = 0; c < KCH; ++c) acc[q][c] = make_float4(0.f, 0.f, 0.f, 0.f);
  }

  const int nchunks = (p.n_str + kStreamRows - 1) / kStreamRows;
  const int ch_begin = blockIdx.y * p.chunks_per_split;
  const int ch_end = min(nchunks, ch_begin + p.chunks_per_split);

  for (int ch = ch_begin; ch < ch_end; ++ch) {
    const int base = ch * kStreamRows;
    __syncthreads();   // previous chunk fully consumed
    for (int v = tid; v < kStreamRows * (ROWLEN >> 2); v += kThreads) {
      const int t = v / (ROWLEN >> 2), col = (v % (ROWLEN >> 2)) << 2;
      const int row = base + t;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < p.n_str) val = ld4(p.str + (size_t)row * D, col, D, vec_str);
      *reinterpret_cast<float4*>(&stage[(size_t)t * ROWLEN + col]) = val;
    }
    __syncthreads();

    float dot[R];
    RedT<0, R, KCH>::run(a, stage, 0, lane, dot);

    const int k = base + lane;            // stream row handled by this lane
    const bool valid = k < p.n_str;
    float gq[R];                          // BWD: w * G (off-diagonal) for (owner q, stream k)

    if (MODE == MODE_BWD_DC) {
      // owner = centroid (global index own0+q), stream = local utterance row k
      float lse_r = 0.f, g_r = g; int jg_r = -2;
      if (valid) {
        lse_r = __ldg(p.row_stat + k); jg_r = p.spk_offset + k / p.M;
        if (RG) g_r = __ldg(p.grad_rows + k);
      }
#pragma unroll
      for (int q = 0; q < R; ++q) {
        const float S = fmaf(w, dot[q] + eps, b);
        const bool off = valid && (jg_r != own0 + q);
        gq[q] = off ? w * g_r * expf(S - lse_r) : 0.f;
      }
    } else {
#pragma unroll
      for (int q = 0; q < R; ++q) {
        const bool diag = (k == jg[q]);
        const float cosv = (diag ? cd[q] : dot[q]) + eps;       // s3:78-79
        const float S = fmaf(w, cosv, b);                       // s3:27
        if (MODE == MODE_FWD) {
          if (p.sim_out != nullptr && valid && own0 + q < p.n_own)
            p.sim_out[(size_t)(own0 + q) * p.n_str + k] = cosv;
          if (VARIANT == GE2E_SOFTMAX) {
            if (valid && !diag) {   // off-diagonal running state; the diagonal joins in the epilogue
              const float mn = fmaxf(m_run[q], S);
              l_run[q] = l_run[q] * expf(m_run[q] - mn) + expf(S - mn);
              m_run[q] = mn;
            }
          } else {
            if (valid && !diag && S > best[q]) { best[q] = S; bestk[q] = k; }
          }
        } else {  // MODE_BWD_DE (softmax only)
          const float pr = valid ? expf(S - lse[q]) : 0.f;
          const float G = gr[q] * (diag ? -qd[q] : pr);     // own speaker: p_jj - 1 = -q, no cancellation
          dw_acc = fmaf(G, cosv, dw_acc);
          gq[q] = (valid && !diag) ? w * G : 0.f;
        }
      }
    }

    if (MODE != MODE_FWD) {
#pragma unroll 4
      for (int t = 0; t < kStreamRows; ++t) {
        float s[R];
#pragma unroll
        for (int q = 0; q < R; ++q) s[q] = __shfl_sync(0xffffffffu, gq[q], t);
#pragma unroll
        for (int c = 0; c < KCH; ++c) {
          const float4 bv = *reinterpret_cast<const float4*>(&stage[(size_t)t * ROWLEN + c * 128 + (lane << 2)]);
#pragma unroll
          for (int q = 0; q < R; ++q) {
            acc[q][c].x = fmaf(s[q], bv.x, acc[q][c].x);
            acc[q][c].y = fmaf(s[q], bv.y, acc[q][c].y);
            acc[q][c].z = fmaf(s[q], bv.z, acc[q][c].z);
            acc[q][c].w = fmaf(s[q], bv.w, acc[q][c].w);
          }
        }
      }
    }
  }

  // ---------------- epilogue ----------------
  if (MODE == MODE_FWD) {
    float loss_part = 0.f;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const int row = own0 + q;
      const float Sd = fmaf(w, cd[q] + eps, b);
      float per, stat; int ks = -1;
      float aux = 0.f;
      if (VARIANT == GE2E_SOFTMAX) {
        const float mx = fmaxf(warp_max(m_run[q]), Sd);
        const float loff = warp_sum(l_run[q] == 0.f ? 0.f : l_run[q] * expf(m_run[q] - mx));
        close_softmax_row(mx, loff, Sd, eps, stat, aux, per);   // s3:120-121 without overflow
      } else {
        float bv = best[q]; int bk = bestk[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
          if (ov > bv || (ov == bv && ok < bk)) { bv = ov; bk = ok; }
        }
        const float sp = 1.f / (1.f + expf(-Sd));
        per = 1.f - sp;
        stat = bv;
        if (bk != INT_MAX) { ks = bk; per += 1.f / (1.f + expf(-bv)); }
      }
      if (lane == 0 && row < p.n_own) {
        p.row_stat_out[row] = stat;
        if (p.row_aux_out != nullptr) p.row_aux_out[row] = aux;
        if (VARIANT == GE2E_CONTRAST && p.kstar_out != nullptr) p.kstar_out[row] = ks;   // softmax: buffer may be a dummy
        if (p.per_row_out != nullptr) p.per_row_out[row] = per;
        loss_part += per;
      }
    }
    const float tot = block_sum(loss_part, red);
    if (tid == 0) atomicAdd(p.loss_accum, tot);
  } else if (MODE == MODE_BWD_DE) {
    const bool vec_out = is_vec(p.acc_out, D);
    float db_part = 0.f;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const int row = own0 + q;
      if (row < p.n_own) {
#pragma unroll
        for (int c = 0; c < KCH; ++c)
          st4(p.acc_out + (size_t)row * D, (lane << 2) + c * 128, D, vec_out, acc[q][c]);
        // db = sum_k G = -g * eps / (sum exp + eps): closed form (SURVEY 8(a-bis) item 12)
        if (lane == 0) db_part -= gr[q] * eps * expf(-lse[q]);
      }
    }
    const float dw_tot = block_sum(dw_acc, red);
    const float db_tot = block_sum(db_part, red);
    if (tid == 0) { atomicAdd(p.dwdb + 0, dw_tot); atomicAdd(p.dwdb + 1, db_tot); }
  } else {  // MODE_BWD_DC
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const int row = own0 + q;
      if (row < p.n_own) {
        float* out = p.acc_out + (size_t)row * D;
#pragma unroll
        for (int c = 0; c < KCH; ++c) {
          const int col = (lane << 2) + c * 128;
          if (col + 0 < D) atomicAdd(out + col + 0, acc[q][c].x);
          if (col + 1 < D) atomicAdd(out + col + 1, acc[q][c].y);
          if (col + 2 < D) atomicAdd(out + col + 2, acc[q][c].z);
          if (col + 3 < D) atomicAdd(out + col + 3, acc[q][c].w);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// contrast backward: G has two non-zeros per row (the diagonal and k*): gather / scatter.
// grid = ceil(U_local / 8), block = 256 (one warp per utterance row)
// gp: the upstream gradient -- one scalar, or (RG) one per utterance row
// ------------------------------------------------------------------------------------------
template <bool RG = false>
__global__ void __launch_bounds__(kThreads)
contrast_bwd_kernel(const float* __restrict__ e_hat, const float* __restrict__ c_hat_all,
                    const float* __restrict__ cos_diag, const float* __restrict__ row_stat,
                    const int32_t* __restrict__ kstar, int U, int D, const float* __restrict__ wp,
                    const float* __restrict__ bp, float eps, const float* __restrict__ gp,
                    float* __restrict__ dE_hat, float* __restrict__ dC_hat, float* __restrict__ dwdb) {
  __shared__ float red[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int r = blockIdx.x * kWarps + wid;
  const float w = __ldg(wp), b = __ldg(bp), g0 = RG ? 0.f : __ldg(gp);
  float dw = 0.f, db = 0.f;
  if (r < U) {
    const float g = RG ? __ldg(gp + r) : g0;
    const float cd = __ldg(cos_diag + r) + eps;
    const float sp = 1.f / (1.f + expf(-fmaf(w, cd, b)));
    const float Gp = -g * sp * (1.f - sp);
    const int ks = __ldg(kstar + r);
    float Gn = 0.f, cn = 0.f;
    const float* er = e_hat + (size_t)r * D;
    if (ks >= 0) {
      const float* ck = c_hat_all + (size_t)ks * D;
      float d = 0.f;
      for (int c = lane; c < D; c += 32) d = fmaf(__ldg(er + c), __ldg(ck + c), d);
      cn = warp_sum(d) + eps;
      const float sn = 1.f / (1.f + expf(-__ldg(row_stat + r)));
      Gn = g * sn * (1.f - sn);
      const float wg = w * Gn;
      for (int c = lane; c < D; c += 32) {
        dE_hat[(size_t)r * D + c] = wg * __ldg(ck + c);
        atomicAdd(dC_hat + (size_t)ks * D + c, wg * __ldg(er + c));
      }
    } else {
      for (int c = lane; c < D; c += 32) dE_hat[(size_t)r * D + c] = 0.f;
    }
    if (lane == 0) { dw = Gp * cd + Gn * cn; db = Gp + Gn; }
  }
  const float dwt = block_sum(dw, red);
  const float dbt = block_sum(db, red);
  if (tid == 0) { atomicAdd(dwdb + 0, dwt); atomicAdd(dwdb + 1, dbt); }
}

// contrast_bwd_kernel, speaker-sharded over peer memory: row r's w G_n e_hat_r is added straight into the owner
// rank's dC_local row (centroid k* lives at row k* % peer_rows of rank k* / peer_rows) instead of a full-height
// dC_hat partial.  The adds are system-scope reductions performed at the owner's memory, since every rank adds into
// the same rows at once.  VEC (D % 4 == 0, every row 16-byte aligned): red.global.add.v4.f32, one float4 a lane per
// 128 columns.  dE_hat and {dw, db} as in contrast_bwd_kernel.
struct PeerRows { float* p[GE2E_MAX_PEERS]; };

template <bool RG, bool VEC>
__global__ void __launch_bounds__(kThreads)
contrast_bwd_peers_kernel(const float* __restrict__ e_hat, const float* __restrict__ c_hat_all,
                          const float* __restrict__ cos_diag, const float* __restrict__ row_stat,
                          const int32_t* __restrict__ kstar, int U, int D, const float* __restrict__ wp,
                          const float* __restrict__ bp, float eps, const float* __restrict__ gp,
                          float* __restrict__ dE_hat, PeerRows owner, int peer_rows, float* __restrict__ dwdb) {
  __shared__ float red[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int r = blockIdx.x * kWarps + wid;
  const float w = __ldg(wp), b = __ldg(bp), g0 = RG ? 0.f : __ldg(gp);
  float dw = 0.f, db = 0.f;
  if (r < U) {
    const float g = RG ? __ldg(gp + r) : g0;
    const float cd = __ldg(cos_diag + r) + eps;
    const float sp = 1.f / (1.f + expf(-fmaf(w, cd, b)));
    const float Gp = -g * sp * (1.f - sp);
    const int ks = __ldg(kstar + r);
    float Gn = 0.f, cn = 0.f;
    const float* er = e_hat + (size_t)r * D;
    float* de = dE_hat + (size_t)r * D;
    if (ks >= 0) {
      const float* ck = c_hat_all + (size_t)ks * D;
      const int o = ks / peer_rows;
      float* dst = owner.p[0];          // owner.p[o] by selects: a dynamic index would copy the array to local memory
#pragma unroll
      for (int q = 1; q < GE2E_MAX_PEERS; ++q)
        if (q == o) dst = owner.p[q];
      dst += (size_t)(ks - o * peer_rows) * D;
      const float sn = 1.f / (1.f + expf(-__ldg(row_stat + r)));
      Gn = g * sn * (1.f - sn);
      const float wg = w * Gn;
      float d = 0.f;
      if (VEC) {
        const float4* er4 = reinterpret_cast<const float4*>(er);
        const float4* ck4 = reinterpret_cast<const float4*>(ck);
        for (int c = lane; c < (D >> 2); c += 32) {
          const float4 e = __ldg(er4 + c), k = __ldg(ck4 + c);
          d = fmaf(e.x, k.x, fmaf(e.y, k.y, fmaf(e.z, k.z, fmaf(e.w, k.w, d))));
          reinterpret_cast<float4*>(de)[c] = make_float4(wg * k.x, wg * k.y, wg * k.z, wg * k.w);
          asm volatile("red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * c),
                       "f"(wg * e.x), "f"(wg * e.y), "f"(wg * e.z), "f"(wg * e.w)
                       : "memory");
        }
      } else {
        for (int c = lane; c < D; c += 32) {
          d = fmaf(__ldg(er + c), __ldg(ck + c), d);
          de[c] = wg * __ldg(ck + c);
          asm volatile("red.relaxed.sys.global.add.f32 [%0], %1;" ::"l"(dst + c), "f"(wg * __ldg(er + c)) : "memory");
        }
      }
      cn = warp_sum(d) + eps;
    } else {
      for (int c = lane; c < D; c += 32) de[c] = 0.f;
    }
    if (lane == 0) { dw = Gp * cd + Gn * cn; db = Gp + Gn; }
  }
  const float dwt = block_sum(dw, red);
  const float dbt = block_sum(db, red);
  if (tid == 0) { atomicAdd(dwdb + 0, dwt); atomicAdd(dwdb + 1, dbt); }
}

// ------------------------------------------------------------------------------------------
// K4: finalize.  grid = n_local, block = 256, dynamic smem = (2*M + 2) * Dp floats.
// ------------------------------------------------------------------------------------------
// Body shared by finalize_kernel and the fused small-batch kernel: speaker j, block of kThreads
// threads, `smem` = (2 M + 2) * Dp floats.  dE_hat / dC_hat are read with plain loads (the fused
// kernel reads what its own block has just written).
// REUSE_E: sE already holds the speaker's raw rows (prep_body staged them at the same place earlier in this kernel).
// RG: the upstream gradient of logical row r is g_rows[r] (g unused); where bwd_rows already folded it into dE_hat
// (row_scale == nullptr) it only enters the diagonal term.
template <bool REUSE_E = false, typename TE = float, typename TD = float, bool RG = false>
__device__ __forceinline__ void finalize_body(const TE* __restrict__ E, const float* dE_hat, const float* dC_hat,
                                              const float* cos_diag, const float* row_stat, const float* row_aux,
                                              const float* row_scale, int j, int M, int D, int Dp, float w, float b,
                                              float g, float eps,
                                              int variant, TD* __restrict__ dE, const int32_t* __restrict__ idx,
                                              float* smem, const float* __restrict__ g_rows = nullptr) {
  __shared__ float red[kWarps];
  __shared__ float s_bc[2];
  float* sE = smem;                          // [M][Dp] raw embeddings -> later de (gradient through e_hat)
  float* sU = sE + (size_t)M * Dp;           // [M][Dp] du rows
  float* sS = sU + (size_t)M * Dp;           // [Dp] column sums of E, later sum_i du
  float* sB = sS + Dp;                       // [Dp] dc_j / M
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const bool vec_g = is_vec(dE_hat, D), vec_o = is_vec(dE, D);

  if (!REUSE_E) stage_rows(E, idx, j, M, D, Dp, sE);
  for (int d = tid; d < Dp; d += kThreads) {
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += sE[(size_t)i * Dp + d];
    sS[d] = s;
  }
  __syncthreads();

  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  {
    float ss = 0.f, pr = 0.f;
    for (int d = tid; d < D; d += kThreads) {
      ss = fmaf(sS[d], sS[d], ss);
      pr = fmaf(sS[d], REUSE_E ? __ldcg(dC_hat + (size_t)j * D + d) : dC_hat[(size_t)j * D + d], pr);
    }
    const float sst = block_sum(ss, red);
    const float prt = block_sum(pr, red);
    if (tid == 0) { s_bc[0] = sst; s_bc[1] = prt; }
    __syncthreads();
    const float2 k = centroid_jacobian(s_bc[0], s_bc[1], inv_m);
    for (int d = tid; d < Dp; d += kThreads) {
      float v = 0.f;
      if (d < D) v = (REUSE_E ? __ldcg(dC_hat + (size_t)j * D + d) : dC_hat[(size_t)j * D + d]) * k.x - sS[d] * k.y;
      sB[d] = v;
    }
  }
  __syncthreads();

  for (int i = wid; i < M; i += kWarps) {
    const int r = j * M + i;
    float ne2 = 0.f, nd2 = 0.f, ed = 0.f, eg = 0.f;
    const float* gh = dE_hat + (size_t)r * D;
    const float gr = RG ? __ldg(g_rows + r) : g;
    // tensor-core softmax path: dE_hat holds un-normalised rows, the true row is g * row_scale[r] times it
    const float gsc = row_scale != nullptr ? gr * row_scale[r] : 1.f;
    for (int d = lane << 2; d < Dp; d += 128) {
      const float4 e = *reinterpret_cast<const float4*>(&sE[(size_t)i * Dp + d]);
      const float4 s = *reinterpret_cast<const float4*>(&sS[d]);
      const float4 gv = ld4_plain(gh, d, D, vec_g);
      const float4 dv = make_float4(s.x - e.x, s.y - e.y, s.z - e.z, s.w - e.w);
      ne2 += dot4(e, e); nd2 += dot4(dv, dv); ed += dot4(e, dv); eg += dot4(e, gv);
    }
    const RowNorms n = row_norms(warp_sum(ne2), warp_sum(nd2), warp_sum(ed), inv_m1);
    const float dd = diag_term(variant, gr, variant == GE2E_SOFTMAX ? row_aux[r] : cos_diag[r], w, b, eps);
    const RowJacobian J = row_jacobian(n, warp_sum(eg) * gsc, gsc, dd, inv_m1);
    for (int d = lane << 2; d < Dp; d += 128) {
      const float4 e = *reinterpret_cast<const float4*>(&sE[(size_t)i * Dp + d]);
      const float4 s = *reinterpret_cast<const float4*>(&sS[d]);
      const float4 gv = ld4_plain(gh, d, D, vec_g);
      const float ev[4] = {e.x, e.y, e.z, e.w}, sv[4] = {s.x, s.y, s.z, s.w}, gg[4] = {gv.x, gv.y, gv.z, gv.w};
      float de[4], du[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        de[t] = J.de(ev[t], sv[t] - ev[t], gg[t]);
        du[t] = J.du(ev[t], sv[t] - ev[t]);
      }
      // each (i, d) slot is read and then overwritten by the same single lane: no cross-lane hazard
      // (and no __syncwarp here: for D < 128 only some lanes enter this loop)
      *reinterpret_cast<float4*>(&sU[(size_t)i * Dp + d]) = make_float4(du[0], du[1], du[2], du[3]);
      *reinterpret_cast<float4*>(&sE[(size_t)i * Dp + d]) = make_float4(de[0], de[1], de[2], de[3]);
    }
  }
  __syncthreads();   // sS (sums of E) no longer needed after this point
  for (int d = tid; d < Dp; d += kThreads) {
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += sU[(size_t)i * Dp + d];
    sS[d] = s;
  }
  __syncthreads();
  for (int v = tid; v < M * (Dp >> 2); v += kThreads) {
    const int i = v / (Dp >> 2), col = (v % (Dp >> 2)) << 2;
    const float4 de = *reinterpret_cast<const float4*>(&sE[(size_t)i * Dp + col]);
    const float4 du = *reinterpret_cast<const float4*>(&sU[(size_t)i * Dp + col]);
    const float4 sd = *reinterpret_cast<const float4*>(&sS[col]);
    const float4 bc = *reinterpret_cast<const float4*>(&sB[col]);
    float4 o;
    o.x = de.x + bc.x + (sd.x - du.x) * inv_m1;
    o.y = de.y + bc.y + (sd.y - du.y) * inv_m1;
    o.z = de.z + bc.z + (sd.z - du.z) * inv_m1;
    o.w = de.w + bc.w + (sd.w - du.w) * inv_m1;
    st4e(dE + phys_row(idx, (size_t)j * M + i) * D, col, D, vec_o, o);
  }
}

// gp: the upstream gradient -- one scalar, or (RG) one per logical utterance row
template <typename TE, typename TD, bool RG = false>
__global__ void __launch_bounds__(kThreads)
finalize_kernel(const TE* __restrict__ E, const float* __restrict__ dE_hat,
                const float* __restrict__ dC_hat, const float* __restrict__ cos_diag,
                const float* __restrict__ row_stat, const float* __restrict__ row_aux,
                const float* __restrict__ row_scale, int M, int D, int Dp,
                const float* __restrict__ wp, const float* __restrict__ bp, float eps, int variant,
                const float* __restrict__ gp, TD* __restrict__ dE, const int32_t* __restrict__ idx) {
  extern __shared__ __align__(16) float smem[];
  finalize_body<false, TE, TD, RG>(E, dE_hat, dC_hat, cos_diag, row_stat, row_aux, row_scale, blockIdx.x, M, D, Dp, __ldg(wp),
                                  __ldg(bp), RG ? 0.f : __ldg(gp), eps, variant, dE, idx, smem, gp);
}


// ------------------------------------------------------------------------------------------
// K4 (fast path): one WARP per speaker (M <= 32, D = 128 KCH, aligned), same math as
// finalize_kernel below without shared memory / block barriers / divisions.  Three passes over
// the speaker's rows (the 2nd and 3rd hit L1): column sums; per-row scalars + sum_i du_i;
// outputs.  Row i's scalars live in lane i between the passes.
// ------------------------------------------------------------------------------------------
template <int KCH, typename TE, typename TD, bool RG = false>
__global__ void __launch_bounds__(kPrepWarps * 32)
finalize_warp_kernel(const TE* __restrict__ E, const float* __restrict__ dE_hat,
                     const float* __restrict__ dC_hat, const float* __restrict__ cos_diag,
                     const float* __restrict__ row_aux, const float* __restrict__ row_scale, int n_local, int M,
                     const float* __restrict__ wp, const float* __restrict__ bp, float eps, int variant,
                     const float* __restrict__ gp, TD* __restrict__ dE, const int32_t* __restrict__ idx) {
  constexpr int D = KCH * 128;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int j = blockIdx.x * kPrepWarps + wid;
  pdl_wait();        // launched with the PDL attribute: dE_hat / dC_hat come from the preceding grids
  pdl_trigger();     // the next step's prep may be scheduled (it waits for this grid before touching memory)
  if (j >= n_local) return;
  const float w = __ldg(wp), b = __ldg(bp), g = RG ? 0.f : __ldg(gp);
  auto rowp = [&](int i) {      // + c * 32 vectors per 128-column chunk
    return reinterpret_cast<const vec4_t<TE>*>(E + phys_row(idx, (size_t)j * M + i) * D) + lane;
  };
  const float4* Gj = reinterpret_cast<const float4*>(dE_hat + (size_t)j * M * D) + lane;
  float4 s[KCH];
#pragma unroll
  for (int c = 0; c < KCH; ++c) s[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i0 = 0; i0 < M; i0 += kRowBatch) {
    float4 v[kRowBatch][KCH];
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r)
#pragma unroll
      for (int c = 0; c < KCH; ++c)
        v[r][c] = (i0 + r < M) ? ldg4v<TE>(rowp(i0 + r) + c * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r)
#pragma unroll
      for (int c = 0; c < KCH; ++c) {
        s[c].x += v[r][c].x; s[c].y += v[r][c].y; s[c].z += v[r][c].z; s[c].w += v[r][c].w;
      }
  }
  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  float4 bc[KCH];     // dc_j / M
  {
    float4 dch[KCH];
    float ss = 0.f, pr = 0.f;
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      dch[c] = __ldg(reinterpret_cast<const float4*>(dC_hat + (size_t)j * D) + lane + c * 32);
      ss += dot4(s[c], s[c]);
      pr += dot4(s[c], dch[c]);
    }
    const float2 k = centroid_jacobian(warp_sum(ss), warp_sum(pr), inv_m);
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      bc[c].x = dch[c].x * k.x - s[c].x * k.y; bc[c].y = dch[c].y * k.x - s[c].y * k.y;
      bc[c].z = dch[c].z * k.x - s[c].z * k.y; bc[c].w = dch[c].w * k.x - s[c].w * k.y;
    }
  }
  // pass 2: the Jacobian of every row (kept in lane i) and sd = sum_i du_i
  RowJacobian Jl = {0.f, 0.f, 0.f, 0.f, 0.f};     // this lane's row (row index == lane)
  float4 sd[KCH];
#pragma unroll
  for (int c = 0; c < KCH; ++c) sd[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i0 = 0; i0 < M; i0 += kRowBatch) {
    float4 v[kRowBatch][KCH];
    float ne2[kRowBatch], nd2[kRowBatch], ed[kRowBatch], eg[kRowBatch];
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r) {
      ne2[r] = 0.f; nd2[r] = 0.f; ed[r] = 0.f; eg[r] = 0.f;
#pragma unroll
      for (int c = 0; c < KCH; ++c) {
        const bool in = i0 + r < M;
        v[r][c] = in ? ldg4v<TE>(rowp(i0 + r) + c * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 gv = in ? __ldg(Gj + (size_t)(i0 + r) * (D / 4) + c * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 e = v[r][c];
        const float4 d = make_float4(s[c].x - e.x, s[c].y - e.y, s[c].z - e.z, s[c].w - e.w);
        ne2[r] += dot4(e, e); nd2[r] += dot4(d, d); ed[r] += dot4(e, d); eg[r] += dot4(e, gv);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < kRowBatch; ++r) {
        ne2[r] += __shfl_xor_sync(0xffffffffu, ne2[r], o);
        nd2[r] += __shfl_xor_sync(0xffffffffu, nd2[r], o);
        ed[r] += __shfl_xor_sync(0xffffffffu, ed[r], o);
        eg[r] += __shfl_xor_sync(0xffffffffu, eg[r], o);
      }
#pragma unroll
    for (int r = 0; r < kRowBatch; ++r) {
      if (i0 + r < M) {
        const int row = j * M + i0 + r;
        const RowNorms n = row_norms(ne2[r], nd2[r], ed[r], inv_m1);
        const float gr = RG ? __ldcg(gp + row) : g;                 // upstream gradient of this row
        const float dd = diag_term(variant, gr, variant == GE2E_SOFTMAX ? __ldg(row_aux + row) : __ldg(cos_diag + row),
                                   w, b, eps);
        const float gsc = row_scale != nullptr ? gr * __ldcg(row_scale + row) : 1.f;   // un-normalised dE_hat rows
        const RowJacobian J = row_jacobian(n, eg[r] * gsc, gsc, dd, inv_m1);
        if (lane == i0 + r) Jl = J;
#pragma unroll
        for (int c = 0; c < KCH; ++c) {
          const float4 e = v[r][c];
          sd[c].x += J.du(e.x, s[c].x - e.x); sd[c].y += J.du(e.y, s[c].y - e.y);
          sd[c].z += J.du(e.z, s[c].z - e.z); sd[c].w += J.du(e.w, s[c].w - e.w);
        }
      }
    }
  }
  // pass 3: dE_i = de_i + dc_j / M + (sd - du_i) / (M - 1)
  for (int i = 0; i < M; ++i) {
    vec4_t<TD>* Oi = reinterpret_cast<vec4_t<TD>*>(dE + phys_row(idx, (size_t)j * M + i) * D) + lane;
    RowJacobian J;
    J.a_g = __shfl_sync(0xffffffffu, Jl.a_g, i); J.a_e = __shfl_sync(0xffffffffu, Jl.a_e, i);
    J.a_d = __shfl_sync(0xffffffffu, Jl.a_d, i); J.b_e = __shfl_sync(0xffffffffu, Jl.b_e, i);
    J.b_d = __shfl_sync(0xffffffffu, Jl.b_d, i);
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      const float4 e = ldg4v<TE>(rowp(i) + c * 32);
      const float4 gv = __ldg(Gj + (size_t)i * (D / 4) + c * 32);
      const float ev[4] = {e.x, e.y, e.z, e.w}, gg[4] = {gv.x, gv.y, gv.z, gv.w};
      const float sv[4] = {s[c].x, s[c].y, s[c].z, s[c].w}, sdv[4] = {sd[c].x, sd[c].y, sd[c].z, sd[c].w};
      const float bv[4] = {bc[c].x, bc[c].y, bc[c].z, bc[c].w};
      float o[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float d = sv[t] - ev[t];
        o[t] = J.de(ev[t], d, gg[t]) + bv[t] + (sdv[t] - J.du(ev[t], d)) * inv_m1;
      }
      st4vv<TD>(Oi + c * 32, make_float4(o[0], o[1], o[2], o[3]));
    }
  }
}

// ------------------------------------------------------------------------------------------
// K4 (register-resident variant, M <= 16, D = 128 W): W warps per speaker, split over the columns as
// in prep_reg_kernel.  The speaker's E rows are loaded once (before the programmatic-launch wait: E
// is not produced by the preceding grids) and stay in registers; everything the preceding grids
// produced (dE_hat rows, the dC_hat row, the row scalars) is requested right after the wait, in one
// batch; dE_hat rows are read twice (L2 / L1 hits).  Row sums through reduce16_transposed and
// speaker_sum, the per-row Jacobian coefficients are computed lane-parallel (lane l owns row
// rev4(l & 15)) and broadcast; the column sums (s, sum_i du_i) never leave the warp.
//   dE_i = de_i + dc_j / M + (sum_i' du_i' - du_i) / (M - 1)
// ------------------------------------------------------------------------------------------
template <int W, int RR, typename TE, typename TD, bool RG = false>
__global__ void __launch_bounds__(kPrepWarps * 32, kRegBlocksPerSM)
finalize_reg_kernel(const TE* __restrict__ E, const float* __restrict__ dE_hat,
                    const float* __restrict__ dC_hat, const float* __restrict__ cos_diag,
                    const float* __restrict__ row_aux, const float* __restrict__ row_scale, int n_local, int M,
                    const float* __restrict__ wp, const float* __restrict__ bp, float eps, int variant,
                    const float* __restrict__ gp, TD* __restrict__ dE, const int32_t* __restrict__ idx) {
  constexpr int D = W * 128, R = RR;       // rows held in registers (M <= R <= 16)
  static_assert(R <= 16, "reduce16_transposed handles 16 rows");
  static_assert(kPrepWarps % W == 0, "a block holds whole speakers");
  __shared__ float xch[kPrepWarps][6][16];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int j = blockIdx.x * (kPrepWarps / W) + wid / W;
  const int col = 128 * (wid % W) + 4 * lane;     // this lane's four columns of every row
  const bool active = j < n_local;
  float4 v[R];
  // the row index is an input of the whole op as well (never written by the preceding grids)
#pragma unroll
  for (int i = 0; i < R; ++i)
    v[i] = (active && i < M) ? ldg4(E + phys_row(idx, (size_t)j * M + i) * D + col) : make_float4(0.f, 0.f, 0.f, 0.f);
  // what depends on E alone runs before the wait: the column sum s and the partial row sums |e|^2, |s - e|^2,
  // e.(s - e) and |s|^2 (t[1..4]); e.dE_hat and s.dC_hat (t[0], t[5]) follow it
  float4 s = v[0];
#pragma unroll
  for (int i = 1; i < R; ++i) { s.x += v[i].x; s.y += v[i].y; s.z += v[i].z; s.w += v[i].w; }
  float t[6];
  {
    float ne2[16], nd2[16], ed[16];
#pragma unroll
    for (int i = R; i < 16; ++i) { ne2[i] = 0.f; nd2[i] = 0.f; ed[i] = 0.f; }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const float4 e = v[i];
      const float4 d = make_float4(s.x - e.x, s.y - e.y, s.z - e.z, s.w - e.w);
      ne2[i] = dot4(e, e); nd2[i] = dot4(d, d); ed[i] = dot4(e, d);
    }
    t[1] = reduce16_transposed(ne2, lane); t[2] = reduce16_transposed(nd2, lane); t[3] = reduce16_transposed(ed, lane);
    t[4] = warp_sum(dot4(s, s));
  }
  pdl_wait();        // launched with the PDL attribute: dE_hat / dC_hat come from the preceding grids
  pdl_trigger();     // the next step's prep may be scheduled (it waits for this grid before touching memory)
  if (!active) return;     // all W warps of the speaker
  const float w = __ldg(wp), b = __ldg(bp), g = RG ? 0.f : __ldg(gp);
  const int my_row = rev4(lane & 15);
  const int row = j * M + min(my_row, M - 1);     // lanes past row M - 1 hold no row
  const float4 dch = __ldcg(reinterpret_cast<const float4*>(dC_hat + (size_t)j * D + col));
  const float aux = variant == GE2E_SOFTMAX ? __ldcg(row_aux + row) : __ldg(cos_diag + row);
  // un-normalised dE_hat rows (RG: g_r joins below -- loaded here it would be one more register through the sums)
  const float gsc0 = row_scale != nullptr ? (RG ? __ldcg(row_scale + row) : g * __ldcg(row_scale + row)) : 1.f;
  const float* Gj = dE_hat + (size_t)j * M * D + col;
  {
    float eg[16];
#pragma unroll
    for (int i = R; i < 16; ++i) eg[i] = 0.f;
#pragma unroll
    for (int i = 0; i < R; ++i)
      eg[i] = dot4(v[i], (i < M) ? __ldg(reinterpret_cast<const float4*>(Gj + (size_t)i * D)) : make_float4(0.f, 0.f, 0.f, 0.f));
    t[0] = reduce16_transposed(eg, lane);
    t[5] = warp_sum(dot4(s, dch));
  }
  speaker_sum<W>(t, xch, wid, lane);
  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  const float2 k = centroid_jacobian(t[4], t[5], inv_m);
  const float4 bc = make_float4(dch.x * k.x - s.x * k.y, dch.y * k.x - s.y * k.y, dch.z * k.x - s.z * k.y,
                                dch.w * k.x - s.w * k.y);     // dc_j / M
  RowJacobian J;     // this lane's row
  {
    const float gr = RG ? __ldcg(gp + row) : g;                   // upstream gradient of this lane's row
    const float gsc = (RG && row_scale != nullptr) ? gr * gsc0 : gsc0;
    J = row_jacobian(row_norms(t[1], t[2], t[3], inv_m1), t[0] * gsc, gsc, diag_term(variant, gr, aux, w, b, eps),
                     inv_m1);
  }
  float4 sd = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int i = 0; i < R; ++i) {
    if (i < M) {
      const float r_be = __shfl_sync(0xffffffffu, J.b_e, rev4(i)), r_bd = __shfl_sync(0xffffffffu, J.b_d, rev4(i));
      const float4 e = v[i];
      sd.x += r_be * e.x + r_bd * (s.x - e.x); sd.y += r_be * e.y + r_bd * (s.y - e.y);
      sd.z += r_be * e.z + r_bd * (s.z - e.z); sd.w += r_be * e.w + r_bd * (s.w - e.w);
    }
  }
  // dE_i = de_i + bc + (sd - du_i) / (M - 1), with d_i = s - e_i, is k_g gv_i + k_e e_i + k_s s + base:
  // three coefficients per row instead of five
  const float k_s = J.a_d - J.b_d * inv_m1;
  const float k_e = J.a_e - J.b_e * inv_m1 - k_s;
  const float4 base = make_float4(fmaf(sd.x, inv_m1, bc.x), fmaf(sd.y, inv_m1, bc.y), fmaf(sd.z, inv_m1, bc.z),
                                  fmaf(sd.w, inv_m1, bc.w));
#pragma unroll
  for (int i = 0; i < R; ++i) {
    if (i < M) {
      const float r_g = __shfl_sync(0xffffffffu, J.a_g, rev4(i)), r_e = __shfl_sync(0xffffffffu, k_e, rev4(i));
      const float r_s = __shfl_sync(0xffffffffu, k_s, rev4(i));
      const float4 e = v[i];
      const float4 gv = __ldg(reinterpret_cast<const float4*>(Gj + (size_t)i * D));
      const float4 o = make_float4(r_g * gv.x + r_e * e.x + fmaf(r_s, s.x, base.x), r_g * gv.y + r_e * e.y + fmaf(r_s, s.y, base.y),
                                   r_g * gv.z + r_e * e.z + fmaf(r_s, s.z, base.z), r_g * gv.w + r_e * e.w + fmaf(r_s, s.w, base.w));
      st4v(dE + phys_row(idx, (size_t)j * M + i) * D + col, o);
    }
  }
}

// ------------------------------------------------------------------------------------------
// static helpers of the reference class
// ------------------------------------------------------------------------------------------
__global__ void centroids_kernel(const float* __restrict__ E, int M, int D, float* __restrict__ C) {
  const int j = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += __ldg(E + ((size_t)j * M + i) * D + d);
    C[(size_t)j * D + d] = s / (float)M;   // s3:37
  }
}

__global__ void utt_centroids_kernel(const float* __restrict__ E, int M, int D, float* __restrict__ Uc) {
  const int j = blockIdx.x;
  const float m1 = (float)(M - 1);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += __ldg(E + ((size_t)j * M + i) * D + d);
    for (int i = 0; i < M; ++i) {
      const size_t o = ((size_t)j * M + i) * D + d;
      Uc[o] = (s - __ldg(E + o)) / m1;      // s3:111
    }
  }
}

__global__ void normalize_rows_kernel(const float* __restrict__ X, int rows, int D, float* __restrict__ Y) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int r = blockIdx.x * (blockDim.x >> 5) + wid;
  if (r >= rows) return;
  float n2 = 0.f;
  for (int d = lane; d < D; d += 32) { const float v = __ldg(X + (size_t)r * D + d); n2 = fmaf(v, v, n2); }
  n2 = warp_sum(n2);
  const float inv = 1.f / fmaxf(sqrtf(n2), kCosDelta);
  for (int d = lane; d < D; d += 32) Y[(size_t)r * D + d] = __ldg(X + (size_t)r * D + d) * inv;
}

// calc_loss (s3:114-127) on a caller-supplied S[N, M, N]; one warp per row
__global__ void __launch_bounds__(kThreads)
calc_loss_kernel(const float* __restrict__ S, int N, int M, float eps, int variant,
                 float* __restrict__ loss, float* __restrict__ per_row) {
  __shared__ float red[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int r = blockIdx.x * kWarps + wid;
  float per = 0.f;
  if (r < N * M) {
    const int j = r / M;
    const float* row = S + (size_t)r * N;
    const float Sd = __ldg(row + j);
    if (variant == GE2E_SOFTMAX) {
      float mx = -INFINITY;
      for (int k = lane; k < N; k += 32) mx = fmaxf(mx, __ldg(row + k));
      mx = warp_max(mx);
      float l = 0.f;
      for (int k = lane; k < N; k += 32) l += expf(__ldg(row + k) - mx);
      l = warp_sum(l);
      const float lse = (mx > -80.f) ? mx + logf(l + eps * expf(-mx)) : logf(eps + l * expf(mx));
      per = lse - Sd;
    } else {
      float mx = -INFINITY;
      for (int k = lane; k < N; k += 32) if (k != j) mx = fmaxf(mx, __ldg(row + k));
      mx = warp_max(mx);
      per = 1.f - 1.f / (1.f + expf(-Sd));
      if (N > 1) per += 1.f / (1.f + expf(-mx));
    }
    if (lane == 0 && per_row != nullptr) per_row[r] = per;
    if (lane != 0) per = 0.f;
  }
  const float tot = block_sum(per, red);
  if (tid == 0) atomicAdd(loss, tot);
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024)
    GE2E_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return GE2E_OK;
}

template <int MODE, int VARIANT, int KCH, int R, bool RG>
int launch_strip(const StripParams& p, int splits, cudaStream_t st) {
  const size_t smem = (size_t)kStreamRows * KCH * 128 * sizeof(float);
  auto kern = strip_kernel<MODE, VARIANT, KCH, R, RG>;
  int rc = set_smem(kern, smem);
  if (rc != GE2E_OK) return rc;
  dim3 grid((p.n_own + kWarps * R - 1) / (kWarps * R), splits);
  kern<<<grid, kThreads, smem, st>>>(p);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

template <int MODE, int VARIANT, bool RG = false>
int dispatch_strip(const StripParams& p, int splits, cudaStream_t st) {
  const int D = p.D;
  if (D <= 128) return launch_strip<MODE, VARIANT, 1, 4, RG>(p, splits, st);
  if (D <= 256) return launch_strip<MODE, VARIANT, 2, 4, RG>(p, splits, st);   // R = 8 was tried: 1.65 ms vs 1.40 ms at cfg3
  if (D <= 512) return launch_strip<MODE, VARIANT, 4, 2, RG>(p, splits, st);
  if (D <= 1024) return launch_strip<MODE, VARIANT, 8, 1, RG>(p, splits, st);
  return GE2E_ERR_UNSUPPORTED;
}

int rows_per_cta(int D) { return kWarps * (D <= 256 ? 4 : (D <= 512 ? 2 : 1)); }

}  // namespace

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
// The generic prep / finalize kernels hold a speaker's rows in shared memory: (M + 1) and (2 M + 2) rows of Dp
// floats.  The warp kernels that take over for D = 128 / 256 / 512 with aligned rows cover M <= 32 in finalize,
// which is inside this bound at every D they serve, so the bound is the backward's envelope.
constexpr size_t kGenericSmemCap = 200 * 1024;

int finalize_max_rows(int D) {
  if (D < 1 || D > 1024) return 0;
  const size_t row = (size_t)((D + 3) & ~3) * sizeof(float);
  return (int)(kGenericSmemCap / row / 2) - 1;
}

bool warp_path_ok(int D, std::initializer_list<const void*> ptrs) {
  if (D != 128 && D != 256 && D != 512) return false;
  for (const void* q : ptrs)
    if ((reinterpret_cast<uintptr_t>(q) & 15) != 0) return false;
  return true;
}

// rows of E / dE start at multiples of four elements: 16 bytes for fp32, 8 bytes for the half types
template <typename T>
bool rows_vec_ok(const T* p) { return (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(T) - 1)) == 0; }

// f(TE{}) with the element type of E (ge2e_dtype code, checked by the C ABI)
template <typename F>
int with_e_type(int e_dt, F&& f) {
  if (e_dt == GE2E_DT_BF16) return f(__nv_bfloat16{});
  if (e_dt == GE2E_DT_F16) return f(__half{});
  return f(float{});
}
// f(TE{}, TD{}) with the element types of E and dE (dE: fp32 or E's type)
template <typename F>
int with_e_de_types(int e_dt, int de_dt, F&& f) {
  return with_e_type(e_dt, [&](auto te) -> int { return de_dt == GE2E_DT_F32 ? f(te, float{}) : f(te, te); });
}

template <int KCH, typename TE>
void launch_prep_warp(const TE* E, const int32_t* idx, int n_local, int M, int prec, float* e_hat, float* c_hat,
                      float* cos_diag, float* accum, cudaStream_t st) {
  const int grid = (n_local + kPrepWarps - 1) / kPrepWarps;
  if (KCH <= 2 && M <= kRegRows) {
    // the register-resident variant: one warp per 128 columns, only instantiated for D <= 256
    constexpr int W = KCH <= 2 ? KCH : 1, spb = kPrepWarps / W;
    const dim3 g((n_local + spb - 1) / spb), bl(kPrepWarps * 32);
#define GE2E_PREP_REG(RR)                                                                                          \
  (prec == 3 ? launch_pdl(prep_reg_kernel<W, RR, 3, TE>, g, bl, 0, st, true, E, idx, n_local, M, e_hat, c_hat, cos_diag, accum) \
   : prec == 2 ? launch_pdl(prep_reg_kernel<W, RR, 2, TE>, g, bl, 0, st, true, E, idx, n_local, M, e_hat, c_hat, cos_diag, accum) \
   : prec == 1 ? launch_pdl(prep_reg_kernel<W, RR, 1, TE>, g, bl, 0, st, true, E, idx, n_local, M, e_hat, c_hat, cos_diag, accum) \
               : launch_pdl(prep_reg_kernel<W, RR, 0, TE>, g, bl, 0, st, true, E, idx, n_local, M, e_hat, c_hat, cos_diag, accum))
    if (M <= 4) GE2E_PREP_REG(4); else if (M <= 8) GE2E_PREP_REG(8); else if (M <= 12) GE2E_PREP_REG(12); else GE2E_PREP_REG(16);
#undef GE2E_PREP_REG
    return;
  }
  if (prec == 3) launch_pdl(prep_warp_kernel<KCH, 3, TE>, dim3(grid), dim3(kPrepWarps * 32), 0, st, true, E, idx, n_local, M,
                            e_hat, c_hat, cos_diag, accum);
  else if (prec == 2) launch_pdl(prep_warp_kernel<KCH, 2, TE>, dim3(grid), dim3(kPrepWarps * 32), 0, st, true, E, idx, n_local, M,
                            e_hat, c_hat, cos_diag, accum);
  else if (prec == 1) launch_pdl(prep_warp_kernel<KCH, 1, TE>, dim3(grid), dim3(kPrepWarps * 32), 0, st, true, E, idx, n_local,
                                 M, e_hat, c_hat, cos_diag, accum);
  else launch_pdl(prep_warp_kernel<KCH, 0, TE>, dim3(grid), dim3(kPrepWarps * 32), 0, st, true, E, idx, n_local, M,
                  e_hat, c_hat, cos_diag, accum);
}

template <int KCH, bool RG, typename TE, typename TD>
void launch_finalize_warp(const TE* E, const float* dE_hat, const float* dC_hat, const float* cos_diag,
                          const float* row_aux, const float* row_scale, int n_local, int M, const float* w,
                          const float* b, float eps,
                          int variant, const float* g, TD* dE, const int32_t* idx, bool pdl, cudaStream_t st) {
  const int grid = (n_local + kPrepWarps - 1) / kPrepWarps;
  if (KCH <= 2 && M <= kRegRows) {
    constexpr int W = KCH <= 2 ? KCH : 1, spb = kPrepWarps / W;
    const dim3 gr((n_local + spb - 1) / spb), bl(kPrepWarps * 32);
#define GE2E_FIN_REG(RR)                                                                                     \
  launch_pdl(finalize_reg_kernel<W, RR, TE, TD, RG>, gr, bl, 0, st, pdl, E, dE_hat, dC_hat, cos_diag, row_aux, row_scale, n_local, M, \
             w, b, eps, variant, g, dE, idx)
    if (M <= 4) GE2E_FIN_REG(4); else if (M <= 8) GE2E_FIN_REG(8); else if (M <= 12) GE2E_FIN_REG(12); else GE2E_FIN_REG(16);
#undef GE2E_FIN_REG
    return;
  }
  launch_pdl(finalize_warp_kernel<KCH, TE, TD, RG>, dim3(grid), dim3(kPrepWarps * 32), 0, st, pdl, E, dE_hat, dC_hat, cos_diag,
             row_aux, row_scale, n_local, M, w, b, eps, variant, g, dE, idx);
}

template <typename TE>
int simt_prep_t(const TE* E, const int32_t* row_index, int n_local, int M, int D, int prec, float* e_hat,
                float* c_hat_local, float* cos_diag, float* accum, cudaStream_t st) {
  const bool round_tf32_ = prec == 1;
  if (rows_vec_ok(E) && warp_path_ok(D, {e_hat, c_hat_local})) {
    if (D == 128) launch_prep_warp<1>(E, row_index, n_local, M, prec, e_hat, c_hat_local, cos_diag, accum, st);
    else if (D == 256) launch_prep_warp<2>(E, row_index, n_local, M, prec, e_hat, c_hat_local, cos_diag, accum, st);
    else launch_prep_warp<4>(E, row_index, n_local, M, prec, e_hat, c_hat_local, cos_diag, accum, st);
    GE2E_LAUNCHED();
    return GE2E_OK;
  }
  if (prec >= 2) return GE2E_ERR_UNSUPPORTED;     // the fp16 planes are written by the warp kernels only
  const int Dp = (D + 3) & ~3;
  const size_t smem = (size_t)(M + 1) * Dp * sizeof(float);
  if (smem > kGenericSmemCap) return GE2E_ERR_UNSUPPORTED;
  if (round_tf32_) {
    int rc = set_smem(prep_kernel<true, TE>, smem);
    if (rc != GE2E_OK) return rc;
    prep_kernel<true><<<n_local, kThreads, smem, st>>>(E, row_index, M, D, Dp, e_hat, c_hat_local, cos_diag, accum);
  } else {
    int rc = set_smem(prep_kernel<false, TE>, smem);
    if (rc != GE2E_OK) return rc;
    prep_kernel<false><<<n_local, kThreads, smem, st>>>(E, row_index, M, D, Dp, e_hat, c_hat_local, cos_diag, accum);
  }
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_prep(const void* E, int e_dt, const int32_t* row_index, int n_local, int M, int D, int prec, float* e_hat,
              float* c_hat_local, float* cos_diag, float* accum, cudaStream_t st) {
  return with_e_type(e_dt, [&](auto te) -> int {
    using TE = decltype(te);
    return simt_prep_t(static_cast<const TE*>(E), row_index, n_local, M, D, prec, e_hat, c_hat_local, cos_diag, accum, st);
  });
}

int simt_fwd_rows(const RowsArgs& a, float* row_stat, int32_t* row_kstar, float* row_aux, float* loss_accum,
                  float* per_row_out, float* sim_out, cudaStream_t st) {
  StripParams p{};
  p.own = a.e_hat; p.n_own = a.n_local * a.M;
  p.str = a.c_hat_all; p.n_str = a.n_total;
  p.D = a.D; p.M = a.M; p.spk_offset = a.spk_offset;
  p.cos_diag = a.cos_diag; p.w = a.w; p.b = a.b; p.eps = a.eps;
  p.row_stat_out = row_stat; p.kstar_out = row_kstar; p.row_aux_out = row_aux; p.loss_accum = loss_accum;
  p.per_row_out = per_row_out; p.sim_out = sim_out;
  p.chunks_per_split = INT_MAX / 2;
  if (a.variant == GE2E_SOFTMAX) return dispatch_strip<MODE_FWD, GE2E_SOFTMAX>(p, 1, st);
  return dispatch_strip<MODE_FWD, GE2E_CONTRAST>(p, 1, st);
}

int simt_bwd_rows(const RowsArgs& a, const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                  const float* grad_out, const float* grad_rows, float* dE_hat, float* dC_hat_partial,
                  float* dwdb_accum, cudaStream_t st) {
  const int U = a.n_local * a.M;
  // one memset when the caller placed {dw, db} right behind dC_hat_partial, else two
  const size_t dc_elems = (size_t)a.n_total * a.D;
  if (dwdb_accum == dC_hat_partial + dc_elems) {
    GE2E_CUDA_TRY(cudaMemsetAsync(dC_hat_partial, 0, (dc_elems + 2) * sizeof(float), st));
  } else {
    GE2E_CUDA_TRY(cudaMemsetAsync(dC_hat_partial, 0, dc_elems * sizeof(float), st));
    GE2E_CUDA_TRY(cudaMemsetAsync(dwdb_accum, 0, 2 * sizeof(float), st));
  }
  if (a.variant == GE2E_CONTRAST) {
    if (grad_rows != nullptr)
      contrast_bwd_kernel<true><<<(U + kWarps - 1) / kWarps, kThreads, 0, st>>>(
          a.e_hat, a.c_hat_all, a.cos_diag, row_stat, row_kstar, U, a.D, a.w, a.b, a.eps, grad_rows,
          dE_hat, dC_hat_partial, dwdb_accum);
    else
      contrast_bwd_kernel<<<(U + kWarps - 1) / kWarps, kThreads, 0, st>>>(
          a.e_hat, a.c_hat_all, a.cos_diag, row_stat, row_kstar, U, a.D, a.w, a.b, a.eps, grad_out,
          dE_hat, dC_hat_partial, dwdb_accum);
    GE2E_LAUNCHED();
    return GE2E_OK;
  }
  StripParams p{};
  p.D = a.D; p.M = a.M; p.spk_offset = a.spk_offset;
  p.cos_diag = a.cos_diag; p.row_stat = row_stat; p.row_aux = row_aux; p.w = a.w; p.b = a.b; p.grad_out = grad_out;
  p.grad_rows = grad_rows; p.eps = a.eps;
  const bool rg = grad_rows != nullptr;
  // dE_hat: owner = utterances, stream = centroids
  p.own = a.e_hat; p.n_own = U; p.str = a.c_hat_all; p.n_str = a.n_total;
  p.acc_out = dE_hat; p.dwdb = dwdb_accum; p.chunks_per_split = INT_MAX / 2;
  int rc = rg ? dispatch_strip<MODE_BWD_DE, GE2E_SOFTMAX, true>(p, 1, st) : dispatch_strip<MODE_BWD_DE, GE2E_SOFTMAX>(p, 1, st);
  if (rc != GE2E_OK) return rc;
  // dC_hat: owner = centroids, stream = utterances, stream range split across blockIdx.y
  p.own = a.c_hat_all; p.n_own = a.n_total; p.str = a.e_hat; p.n_str = U;
  p.acc_out = dC_hat_partial; p.dwdb = nullptr;
  const int own_ctas = (a.n_total + rows_per_cta(a.D) - 1) / rows_per_cta(a.D);
  const int nchunks = (U + kStreamRows - 1) / kStreamRows;
  int splits = (2 * 148 + own_ctas - 1) / own_ctas;        // aim at ~2 waves of 148 SMs
  splits = max(1, min(splits, nchunks));
  p.chunks_per_split = (nchunks + splits - 1) / splits;
  splits = (nchunks + p.chunks_per_split - 1) / p.chunks_per_split;
  return rg ? dispatch_strip<MODE_BWD_DC, GE2E_SOFTMAX, true>(p, splits, st)
            : dispatch_strip<MODE_BWD_DC, GE2E_SOFTMAX>(p, splits, st);
}

int simt_contrast_bwd_rows_peers(const RowsArgs& a, const float* row_stat, const int32_t* row_kstar,
                                 const float* grad_out, const float* grad_rows, float* dE_hat, float* dwdb_accum,
                                 float* const* dC_owner, int n_ranks, cudaStream_t st) {
  const int U = a.n_local * a.M, grid = (U + kWarps - 1) / kWarps, peer_rows = a.n_total / n_ranks;
  PeerRows o{};
  for (int r = 0; r < n_ranks; ++r) o.p[r] = dC_owner[r];
  const bool vec = a.D % 4 == 0 && rows_vec_ok(a.e_hat) && rows_vec_ok(a.c_hat_all) && rows_vec_ok(dE_hat);
  const float* g = grad_rows != nullptr ? grad_rows : grad_out;
  GE2E_CUDA_TRY(cudaMemsetAsync(dwdb_accum, 0, 2 * sizeof(float), st));
#define GE2E_CONTRAST_PEERS(RG, VEC)                                                                              \
  contrast_bwd_peers_kernel<RG, VEC><<<grid, kThreads, 0, st>>>(a.e_hat, a.c_hat_all, a.cos_diag, row_stat, row_kstar, \
                                                                U, a.D, a.w, a.b, a.eps, g, dE_hat, o, peer_rows,     \
                                                                dwdb_accum)
  if (grad_rows != nullptr) {
    if (vec) GE2E_CONTRAST_PEERS(true, true); else GE2E_CONTRAST_PEERS(true, false);
  } else {
    if (vec) GE2E_CONTRAST_PEERS(false, true); else GE2E_CONTRAST_PEERS(false, false);
  }
#undef GE2E_CONTRAST_PEERS
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// RG: grad_out is the upstream gradient per logical utterance row
template <bool RG, typename TE, typename TD>
int simt_bwd_finalize_t(const TE* E, const int32_t* row_index, const float* dE_hat, const float* dC_hat_local,
                        const float* cos_diag, const float* row_stat, const float* row_aux, const float* row_scale,
                        int n_local, int M, int D, const float* w, const float* b, float eps, int variant,
                        const float* grad_out, TD* dE, bool pdl, cudaStream_t st) {
  if (M <= 32 && rows_vec_ok(E) && rows_vec_ok(dE) && warp_path_ok(D, {dE_hat, dC_hat_local})) {
    if (D == 128) launch_finalize_warp<1, RG>(E, dE_hat, dC_hat_local, cos_diag, row_aux, row_scale, n_local, M, w, b, eps, variant, grad_out, dE, row_index, pdl, st);
    else if (D == 256) launch_finalize_warp<2, RG>(E, dE_hat, dC_hat_local, cos_diag, row_aux, row_scale, n_local, M, w, b, eps, variant, grad_out, dE, row_index, pdl, st);
    else launch_finalize_warp<4, RG>(E, dE_hat, dC_hat_local, cos_diag, row_aux, row_scale, n_local, M, w, b, eps, variant, grad_out, dE, row_index, pdl, st);
    GE2E_LAUNCHED();
    return GE2E_OK;
  }
  const int Dp = (D + 3) & ~3;
  if (M > finalize_max_rows(D)) return GE2E_ERR_UNSUPPORTED;
  const size_t smem = (size_t)(2 * M + 2) * Dp * sizeof(float);
  int rc = set_smem(finalize_kernel<TE, TD, RG>, smem);
  if (rc != GE2E_OK) return rc;
  finalize_kernel<TE, TD, RG><<<n_local, kThreads, smem, st>>>(E, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, row_scale, M, D,
                                                   Dp, w, b, eps, variant, grad_out, dE, row_index);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_bwd_finalize(const void* E, int e_dt, const int32_t* row_index, const float* dE_hat, const float* dC_hat_local,
                      const float* cos_diag, const float* row_stat, const float* row_aux, const float* row_scale,
                      int n_local, int M, int D, const float* w, const float* b, float eps, int variant,
                      const float* grad_out, const float* grad_rows, void* dE, int de_dt, bool pdl,
                      cudaStream_t st) {
  return with_e_de_types(e_dt, de_dt, [&](auto te, auto td) -> int {
    using TE = decltype(te);
    using TD = decltype(td);
    if (grad_rows != nullptr)
      return simt_bwd_finalize_t<true>(static_cast<const TE*>(E), row_index, dE_hat, dC_hat_local, cos_diag, row_stat,
                                       row_aux, row_scale, n_local, M, D, w, b, eps, variant, grad_rows,
                                       static_cast<TD*>(dE), pdl, st);
    return simt_bwd_finalize_t<false>(static_cast<const TE*>(E), row_index, dE_hat, dC_hat_local, cos_diag, row_stat,
                                      row_aux, row_scale, n_local, M, D, w, b, eps, variant, grad_out,
                                      static_cast<TD*>(dE), pdl, st);
  });
}

// ------------------------------------------------------------------------------------------
// Small batches (the reference's own training / test shapes: N = 64 x M = 10, N = 4 x M = 8): the
// whole fwd+bwd step as ONE kernel.  At these sizes the five-kernel pipeline is pure launch latency
// (cfg2: 52 us for 63 MFLOP), so one CTA per speaker runs every stage, separated by two grid-wide
// barriers (all N <= 128 CTAs are co-resident: one per SM):
//   1  prep_body: e_hat, c_hat_j, cos_diag of the speaker's M rows                     | barrier
//   2  all N c_hat rows -> shared memory; cos / S of the speaker's M x N block; row softmax
//      (or contrast arg-max), loss, dw, db; w G kept in shared memory; dE_hat rows = (wG) C_hat;
//      this speaker's contribution (wG)^T E_hat to every centroid -> workspace [j][k][D]   | barrier
//   3  dC_hat_j = sum over speakers of their contribution to centroid j (fixed order:
//      deterministic); finalize_body: diagonal term, Jacobians, fan-out -> dE
// Same arithmetic as the pipeline's kernels (shared bodies / helpers), fp32 throughout.
//
// Per-utterance losses (reduction "none") learn their upstream gradient g_r only after the forward, so the same
// kernel also runs cut at the seam between the row losses and w G, as two launches (PART):
//   kSmallFwd  1, barrier, 2 up to the row losses: row_stat / row_aux / row_kstar, per_row, loss
//   kSmallBwd  the raw rows re-read; e_hat, c_hat, cos_diag loaded; the cosine block recomputed with the
//              forward's arithmetic (the staged forward stores no cosines either, so both forwards pair with this
//              backward); w G from g_r and the stored row statistics, as the staged kernels form it; rest of 2,
//              barrier, 3.  Its dC_hat rows and {dw, db} are cleared at entry and first added to after the cosine
//              block: one arrival there, its wait in front of the first add.
// ------------------------------------------------------------------------------------------
namespace {

// Up to kSmallMaxN speakers the kernel is correct (tested to 128); it is SELECTED up to kSmallPickN:
// one CTA per speaker serialises the speaker's M x N block, so its advantage over the five-kernel
// pipeline shrinks with N -- 37 -> 9.1 us at the reference's test shape (N = 4, M = 8), 53 -> 19.9 us at its
// training shape (cfg2, N = 64, M = 10; contrast: 30.8 -> 19.7 us; stage timeline: scripts/small_step_trace.py),
// 86 -> 32 us at N = 128, M = 10 (contrast 42 -> 32): selected wherever it is supported.
constexpr int kSmallMaxN = 128, kSmallMaxM = 16, kSmallMaxD = 256, kSmallPickN = 128, kSmallPickNContrast = 128;
constexpr size_t kSmallHeaderBytes = 256;

struct SmallParams {
  const void* E; const int32_t* idx; int M, D, Dp;   // E: element type TE of the kernel
  const float* w; const float* b; float eps;
  const float* grad_out;            // nullable: 1
  float* e_hat; float* c_hat; float* cos_diag; float* row_stat; int32_t* row_kstar; float* row_aux;
  float* per_row;                   // nullable
  float* loss_accum;                // [0] = loss (zeroed here)
  float* dE_hat; float* dC_hat; float* dwdb; void* dE;   // dE: element type TD of the kernel
  int stop;                         // debug, timing only: leave after stage `stop` (0 = run everything)
  int cluster;                      // the grid is ONE thread-block cluster (N <= 8): hardware barriers
  unsigned* ctr;                    // workspace header: {barrier arrivals, exits}; zero on entry, restored
  float* part;                      // workspace: [N][N][D] centroid contributions
  const float* grad_rows;           // kSmallBwd: upstream gradient per logical utterance row (grad_out unused)
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// small_grid_barrier in two halves: after a __syncthreads, thread 0 arrives; release: the block's writes (ordered
// before this thread by the bar.sync) become visible with the arrival
__device__ __forceinline__ void small_grid_arrive(unsigned* ctr) {
  if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
}
// `target` = arrivals expected so far (monotonic counter)
__device__ __forceinline__ void small_grid_wait(const unsigned* ctr, unsigned target) {
  if (threadIdx.x == 0) {
    unsigned long long t0 = 0;
    for (unsigned spins = 0; ld_acquire_u32(ctr) < target; ++spins) {
      if ((spins & 1023u) == 1023u) {               // a missing CTA is a bug: trap instead of hanging the GPU
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t0 == 0) t0 = t;
        else if (t - t0 > 2000000000ull) __trap();
      }
    }
  }
  __syncthreads();
}

// every CTA of the grid arrives
__device__ __forceinline__ void small_grid_barrier(unsigned* ctr, unsigned target) {
  __syncthreads();
  small_grid_arrive(ctr);
  small_grid_wait(ctr, target);
}

// 4 floats of a row that another CTA wrote earlier in this kernel: L2 load (never the L1), tail-safe
__device__ __forceinline__ float4 ld4_cg(const float* row, int col, int D, bool vec) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (vec) { if (col < D) v = __ldcg(reinterpret_cast<const float4*>(row + col)); }
  else {
    if (col + 0 < D) v.x = __ldcg(row + col + 0);
    if (col + 1 < D) v.y = __ldcg(row + col + 1);
    if (col + 2 < D) v.z = __ldcg(row + col + 2);
    if (col + 3 < D) v.w = __ldcg(row + col + 3);
  }
  return v;
}

// MR = M rounded up to a multiple of 4: the cosine block's loops over the speaker's rows are fully
// unrolled without predicates (rows M..MR-1 of the staged e_hat are zero), so the shared-memory loads of
// all rows are issued together instead of one load -> use chain per row.
// PART: kSmallWhole, or one half of the step (kSmallFwd / kSmallBwd, see above)
template <int VARIANT, int MR, typename TE, typename TD, int PART>
__global__ void __launch_bounds__(kThreads, 1)
small_step_kernel(const SmallParams p) {
  const TE* E = static_cast<const TE*>(p.E);
  TD* dE = static_cast<TD*>(p.dE);
  extern __shared__ __align__(16) float smem[];
  __shared__ float red[3 * kWarps];
  __shared__ float s_cd[32];
  __shared__ __align__(8) unsigned long long s_bar;   // bulk-copy completion (stage 2 operands)
  __shared__ float3 s_rsum[16];                       // fast path: |e|^2, |s - e|^2, e.(s - e) per row of the speaker
  __shared__ float s_aux[16];                         // fast path: 1 - p_jj per row
  __shared__ float s_gr[16];                          // kSmallBwd, fast path: g_r per row
  constexpr int R4 = MR / 4;                          // rows per thread where the block splits into 4 row groups
  const int j = blockIdx.x, N = gridDim.x, M = p.M, D = p.D, Dp = p.Dp;
  const int Np = (N + 3) & ~3;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  float* sA = smem;                                   // (2M + 2) Dp: prep_body, later finalize_body
  float* sEh = sA + (size_t)(2 * M + 2) * Dp;         // [MR][Dp] e_hat of this speaker, rows >= M zero
  const int Ds = Dp + 4;                              // row stride of sC: lanes reading different rows hit different banks
  float* sC = sEh + (size_t)MR * Dp;                  // [N][Ds] all c_hat
  float* sG = sC + (size_t)N * Ds;                    // [MR][Np] w * G, zero on the own-speaker column (rows >= M unused)
  float* sCos = sG + (size_t)MR * Np;                 // [MR][Np] cos + eps
  float* sRed = sCos + (size_t)MR * Np;               // [kWarps][MR][32] partial dot products of the cosine block
  if (tid == 0) { ptx::mbar_init(ptx::smem_u32(&s_bar), 1); ptx::fence_mbar_init(); }
  pdl_wait();
  pdl_trigger();
  // debug (GE2E_SMALL_STOP=99, softmax only): SM clock stamps of CTA 0 into the unused row_kstar buffer
#define GE2E_SMALL_STAMP(n) do { if (p.stop == 99 && j == 0 && tid == 0) p.row_kstar[n] = (int)clock(); } while (0)
  GE2E_SMALL_STAMP(0);
  const float w = __ldg(p.w), b = __ldg(p.b), eps = p.eps;
  const float g = p.grad_out != nullptr ? __ldg(p.grad_out) : 1.f;
  if (j == 0 && tid < 4) {
    if (PART != kSmallBwd) p.loss_accum[tid] = 0.f;   // {loss, -, -, -} as prep does
    if (PART != kSmallFwd && tid < 2) p.dwdb[tid] = 0.f;
  }
  // 16-byte rows: the centroid gradient is assembled at the L2 -- every CTA adds its [N][D] share with ONE bulk
  // reduce-add, into rows their owners cleared before the first grid barrier (otherwise: workspace + gather)
  const bool dc_at_l2 = (Dp == D) && is_vec(p.dC_hat, D);
  if (PART != kSmallFwd && dc_at_l2)
    for (int d = tid; d < D; d += kThreads) p.dC_hat[(size_t)j * D + d] = 0.f;

  // ---- 1: this speaker's rows
  // Fast path (whole 16-byte rows of a multiple of 64 columns -- D = 64 / 128 / 192 / 256): the stage bodies shared
  // with the pipeline's kernels (prep_body / finalize_body: a warp per row, M rows in two rounds, every operand
  // through global memory) are replaced by forms that keep the speaker's state in shared memory from here to the
  // last store: a HALF-warp per row (all M <= 16 rows at once), per-row norms computed once, e_hat rows written
  // straight into the stage-2 operand tile, dE_hat rows handed to the Jacobians in shared memory.
  const bool fast = (Dp == D) && (D % 64 == 0) && is_vec(E, D) && is_vec(p.e_hat, D) && is_vec(p.c_hat, D) &&
                    is_vec(p.dE_hat, D) && is_vec(p.dC_hat, D) && is_vec(dE, D);
  float* fE = sA;                                     // [M][Dp] raw rows, later d e (gradient through e_hat)
  float* fS = fE + (size_t)M * Dp;                    // [Dp] column sums of the raw rows, later of d u
  float* fU = fS + Dp;                                // [M][Dp] dE_hat rows, later d u
  float* fB = fU + (size_t)M * Dp;                    // [Dp] dC_hat row, then d c / M
  const int ncol4 = Dp >> 2;
  const int hw = tid >> 4, hl = tid & 15;             // half-warp <-> row
  const float inv_m = 1.f / (float)M, inv_m1 = 1.f / (float)(M - 1);
  float s_norm2 = 0.f, s_mine = 0.f;                  // fast path: |s_j|^2 (every thread), s_j[tid]
  if (fast) {
    for (int i = wid; i < M; i += kWarps) {
      const TE* src = E + phys_row(p.idx, (size_t)j * M + i) * D;
      float4* dst = reinterpret_cast<float4*>(fE + (size_t)i * Dp);
      for (int c4 = lane; c4 < ncol4; c4 += 32) dst[c4] = ldg4(src + 4 * c4);
    }
    for (int v = tid; v < (MR - M) * Dp; v += kThreads) sEh[(size_t)M * Dp + v] = 0.f;
    __syncthreads();
    float spart = 0.f;
    for (int d = tid; d < Dp; d += kThreads) {
      float sum = 0.f;
      for (int i = 0; i < M; ++i) sum += fE[(size_t)i * Dp + d];                 // s3:105
      fS[d] = sum;
      spart = fmaf(sum, sum, spart);
    }
    spart = warp_sum(spart);
    if (lane == 0) red[wid] = spart;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kWarps; ++q) s_norm2 += red[q];
    if (tid < D) {                                     // D <= 256 = block size: one centroid entry per thread
      s_mine = fS[tid];
      if (PART != kSmallBwd) p.c_hat[(size_t)j * D + tid] = s_mine * centroid_scale(s_norm2, inv_m);
    }
    const bool act = hw < M;
    float ne2 = 0.f, nd2 = 0.f, ed = 0.f;
    if (act)
      for (int c4 = hl; c4 < ncol4; c4 += 16) {
        const float4 e = reinterpret_cast<const float4*>(fE + (size_t)hw * Dp)[c4];
        const float4 sv = reinterpret_cast<const float4*>(fS)[c4];
        const float4 dv = make_float4(sv.x - e.x, sv.y - e.y, sv.z - e.z, sv.w - e.w);
        ne2 += dot4(e, e); nd2 += dot4(dv, dv); ed += dot4(e, dv);
      }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      ne2 += __shfl_xor_sync(0xffffffffu, ne2, o);
      nd2 += __shfl_xor_sync(0xffffffffu, nd2, o);
      ed += __shfl_xor_sync(0xffffffffu, ed, o);
    }
    if (PART == kSmallBwd && act && hl == 0) s_rsum[hw] = make_float3(ne2, nd2, ed);   // for the Jacobians only
    if (PART != kSmallBwd && act) {
      const RowNorms n = row_norms(ne2, nd2, ed, inv_m1);
      float4* gdst = reinterpret_cast<float4*>(p.e_hat + ((size_t)j * M + hw) * D);
      for (int c4 = hl; c4 < ncol4; c4 += 16) {
        float4 e = reinterpret_cast<const float4*>(fE + (size_t)hw * Dp)[c4];
        e.x *= n.inv_ne; e.y *= n.inv_ne; e.z *= n.inv_ne; e.w *= n.inv_ne;
        reinterpret_cast<float4*>(sEh + (size_t)hw * Dp)[c4] = e;
        gdst[c4] = e;
      }
      if (hl == 0) { s_cd[hw] = n.cos; p.cos_diag[(size_t)j * M + hw] = n.cos; s_rsum[hw] = make_float3(ne2, nd2, ed); }
    }
  } else if (PART == kSmallBwd) {
    stage_rows(E, p.idx, j, M, D, Dp, sA);            // the raw rows for finalize_body (stage 3)
  } else {
    prep_body<false>(E, p.idx, j, M, D, Dp, p.e_hat, p.c_hat, p.cos_diag, sA);
  }
  GE2E_SMALL_STAMP(1);
  if (p.stop == 1) return;
  do {
  // e_hat / c_hat rows come back through bulk copies (async proxy): order this thread's global writes before them
  asm volatile("fence.proxy.async;" ::: "memory");
  // up to 8 speakers the whole grid is one thread-block cluster: barrier.cluster (release / acquire at cluster
  // scope) instead of an arrival counter polled through the L2
  if (PART == kSmallBwd) {                            // cleared dC_hat rows / {dw, db}: waited for before the adds
    __syncthreads();
    if (p.cluster) ptx::cluster_arrive(); else small_grid_arrive(p.ctr);
  } else if (p.cluster) { __syncthreads(); ptx::cluster_sync_all(); } else small_grid_barrier(p.ctr, (unsigned)N);
  GE2E_SMALL_STAMP(2);
  if (p.stop == 2) break;

  // ---- 2: M x N block of the similarity matrix
  const bool vec_c = is_vec(p.c_hat, D), vec_e = is_vec(p.e_hat, D);
  for (int v = tid; v < (MR - M) * Np; v += kThreads) sG[M * Np + v] = 0.f;    // padding rows of w G: read, never NaN
  if (fast && PART != kSmallBwd) {
    // 16 bytes per cp.async, all of a thread's copies in flight together (a warp takes rows wid, wid + 8, ...):
    // one L2 round trip for the whole centroid matrix; stage 1 left e_hat in sEh and the cosines in s_cd
    for (int k = wid; k < N; k += kWarps) {
      const float4* src = reinterpret_cast<const float4*>(p.c_hat + (size_t)k * D);
      const uint32_t dst = ptx::smem_u32(sC + (size_t)k * Ds);
      for (int c4 = lane; c4 < ncol4; c4 += 32)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (c4 << 4)), "l"(src + c4) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (vec_c && vec_e) {
    // whole rows are 16-byte multiples: one bulk copy per centroid row (the padded row stride keeps 16-byte
    // alignment) and one for the speaker's M contiguous e_hat rows, all counted on one mbarrier
    const uint32_t bar = ptx::smem_u32(&s_bar);
    if (wid == 0) {
      asm volatile("fence.proxy.async;" ::: "memory");     // what the grid barrier acquired -> async proxy
      if (lane == 0) ptx::mbar_expect_tx(bar, static_cast<uint32_t>((N + M) * D * sizeof(float)));
      __syncwarp();
      for (int k = lane; k < N; k += 32)
        ptx::bulk_load_1d(ptx::smem_u32(sC + (size_t)k * Ds), p.c_hat + (size_t)k * D, D * sizeof(float), bar);
      if (lane == 0)
        ptx::bulk_load_1d(ptx::smem_u32(sEh), p.e_hat + (size_t)j * M * D, M * D * sizeof(float), bar);
    }
    for (int v = tid; v < (MR - M) * Dp; v += kThreads) sEh[(size_t)M * Dp + v] = 0.f;
    if (tid < M) s_cd[tid] = p.cos_diag[(size_t)j * M + tid];
    ptx::mbar_wait(bar, 0);
  } else {
    for (int v = tid; v < N * (Dp >> 2); v += kThreads) {
      const int k = v / (Dp >> 2), col = (v % (Dp >> 2)) << 2;
      *reinterpret_cast<float4*>(&sC[(size_t)k * Ds + col]) = ld4_cg(p.c_hat + (size_t)k * D, col, D, vec_c);
    }
    for (int v = tid; v < MR * (Dp >> 2); v += kThreads) {
      const int i = v / (Dp >> 2), col = (v % (Dp >> 2)) << 2;
      *reinterpret_cast<float4*>(&sEh[(size_t)i * Dp + col]) =
          i < M ? ld4_plain(p.e_hat + ((size_t)j * M + i) * D, col, D, vec_e) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (tid < M) s_cd[tid] = p.cos_diag[(size_t)j * M + tid];
  }
  __syncthreads();
  GE2E_SMALL_STAMP(3);
  // thread <-> (centroid kk of KT per pass, column phase dq of DQ = 256 / KT): a thread takes float4 columns dq,
  // dq + DQ, ... of its centroid against ALL the speaker's rows (the centroid row is read once per block, the
  // e_hat columns are warp-wide broadcasts where a warp shares dq), then the DQ partial dot products of every
  // (row, centroid) are added: by shuffles inside a warp (KT < 32), through shared memory across warps, in a fixed
  // order.  Rows M..MR-1 of sEh are zero.  KT: the smallest power of two >= N, between 4 and 64.
  {
    int lkt = 2;
    while ((1 << lkt) < N && lkt < 6) ++lkt;
    const int KT = 1 << lkt, DQ = kThreads >> lkt;
    const int kk = tid & (KT - 1), dq = tid >> lkt;
    const int KW = KT < 32 ? KT : 32;                 // distinct centroids inside one warp
    const int ncol4 = Dp >> 2;
    for (int k0 = 0; k0 < N; k0 += KT) {
      const int k = k0 + kk;
      const float* c = sC + (size_t)(k < N ? k : N - 1) * Ds;
      float acc[MR];
#pragma unroll
      for (int i = 0; i < MR; ++i) acc[i] = 0.f;
#pragma unroll 2
      for (int c4 = dq; c4 < ncol4; c4 += DQ) {
        const float4 cv = *reinterpret_cast<const float4*>(c + (c4 << 2));
#pragma unroll
        for (int i = 0; i < MR; ++i)
          acc[i] += dot4(*reinterpret_cast<const float4*>(sEh + (size_t)i * Dp + (c4 << 2)), cv);
      }
      for (int o = KT; o < 32; o <<= 1) {
#pragma unroll
        for (int i = 0; i < MR; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
      }
      if (lane < KW) {
#pragma unroll
        for (int i = 0; i < MR; ++i) sRed[(wid * MR + i) * 32 + lane] = acc[i];
      }
      __syncthreads();
      // (row i, centroid kk): the warps that hold it are wid = (kk >> 5) + q * wpk, q < nw
      const int wpk = KT > 32 ? KT >> 5 : 1;          // warps that share one dq phase
      const int nw = kWarps / wpk;
      for (int v = tid; v < M * KT; v += kThreads) {
        const int i = v >> lkt, kq = v & (KT - 1), kg = k0 + kq;
        if (kg < N) {
          float t = 0.f;
          for (int q = 0; q < nw; ++q) t += sRed[(((kq >> 5) + q * wpk) * MR + i) * 32 + (kq & 31)];
          sCos[i * Np + kg] = ((kg == j) ? s_cd[i] : t) + eps;                          // s3:78-79
        }
      }
      if (k0 + KT < N) __syncthreads();               // sRed is rewritten by the next pass
    }
  }
  __syncthreads();
  GE2E_SMALL_STAMP(4);
  if (p.stop == 3) break;
  float loss_part = 0.f, dw_part = 0.f, db_part = 0.f;
  for (int i = wid; i < M; i += kWarps) {
    const int r = j * M + i;
    const float cd = sCos[i * Np + j];
    const float Sd = fmaf(w, cd, b);                                                  // s3:27
    const float gr = PART == kSmallBwd ? __ldg(p.grad_rows + r) : g;                 // upstream gradient of the row
    float per, stat, aux = 0.f, dw_i = 0.f, db_i = 0.f;
    int ks = -1;
    if (VARIANT == GE2E_SOFTMAX) {
      // the row's N <= 128 logits stay in registers (4 per lane): one pass for the maximum, one exponential each
      constexpr int kPer = kSmallMaxN / 32;
      float cosv[kPer], ex[kPer];
      float m = -INFINITY;
#pragma unroll
      for (int q = 0; q < kPer; ++q) {
        const int k = lane + 32 * q;
        const bool on = k < N && k != j;
        cosv[q] = on ? sCos[i * Np + k] : 0.f;
        ex[q] = on ? fmaf(w, cosv[q], b) : -INFINITY;
        m = fmaxf(m, ex[q]);
      }
      const float mx = fmaxf(warp_max(m), Sd);
      float l = 0.f;
#pragma unroll
      for (int q = 0; q < kPer; ++q) { ex[q] = expf(ex[q] - mx); l += ex[q]; }      // exp(-inf) = 0 off the row
      const float loff = warp_sum(l);
      if (PART == kSmallBwd) { stat = __ldg(p.row_stat + r); aux = __ldg(p.row_aux + r); per = 0.f; }   // the forward's
      else close_softmax_row(mx, loff, Sd, eps, stat, aux, per);                     // s3:120-121
      if (PART != kSmallFwd) {
        const float sc = gr * expf(mx - stat);          // G_k = g exp(S_k - stat) = sc exp(S_k - mx)
        float dwl = 0.f;
#pragma unroll
        for (int q = 0; q < kPer; ++q) {
          const int k = lane + 32 * q;
          const float G = sc * ex[q];
          dwl = fmaf(G, cosv[q], dwl);
          if (k < N) sG[i * Np + k] = w * G;            // zero on the own-speaker column
        }
        dw_i = warp_sum(dwl) - gr * aux * cd;           // own speaker: G = g (p_jj - 1) = -g aux
        db_i = -gr * eps * expf(-stat);                 // closed form (SURVEY 8(a-bis) item 12)
      }
    } else {
      float bv = -INFINITY; int bk = INT_MAX;
      if (PART == kSmallBwd) {                          // the forward's arg-max and its logit
        bv = __ldg(p.row_stat + r);
        const int k = __ldg(p.row_kstar + r);
        if (k >= 0) bk = k;
      } else {
        for (int k = lane; k < N; k += 32)
          if (k != j) {
            const float S = fmaf(w, sCos[i * Np + k], b);
            if (S > bv) { bv = S; bk = k; }
          }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
          if (ov > bv || (ov == bv && ok < bk)) { bv = ov; bk = ok; }
        }
      }
      const float sp = 1.f / (1.f + expf(-Sd));
      per = 1.f - sp;
      stat = bv;
      const float Gp = -gr * sp * (1.f - sp);
      float Gn = 0.f, cn = 0.f;
      if (bk != INT_MAX) {
        ks = bk;
        const float sn = 1.f / (1.f + expf(-bv));
        per += sn;
        Gn = gr * sn * (1.f - sn);
        cn = sCos[i * Np + bk];
      }
      if (PART != kSmallFwd) {
        for (int k = lane; k < N; k += 32) sG[i * Np + k] = (k == ks) ? w * Gn : 0.f;
        dw_i = Gp * cd + Gn * cn;
        db_i = Gp + Gn;
      }
    }
    if (lane == 0) {
      if (PART != kSmallBwd) p.row_stat[r] = stat;
      if (PART == kSmallWhole || (PART == kSmallFwd && p.row_aux != nullptr)) p.row_aux[r] = aux;
      s_aux[i] = aux;
      if (PART == kSmallBwd) s_gr[i] = gr;
      if (PART != kSmallBwd && VARIANT == GE2E_CONTRAST && p.row_kstar != nullptr) p.row_kstar[r] = ks;
      if (PART != kSmallBwd && p.per_row != nullptr) p.per_row[r] = per;
      loss_part += per; dw_part += dw_i; db_part += db_i;
    }
  }
  if (PART == kSmallBwd) {                             // every CTA has cleared its dC_hat row, CTA 0 {dw, db}
    if (p.cluster) ptx::cluster_wait(); else small_grid_wait(p.ctr, (unsigned)N);
  }
  // lane 0 of every warp holds its rows' {loss, dw, db}: one round through shared memory
  if (lane == 0) { red[wid] = loss_part; red[kWarps + wid] = dw_part; red[2 * kWarps + wid] = db_part; }
  __syncthreads();                                     // sG complete, partial sums staged
  if (tid < 3 && (PART == kSmallWhole || (PART == kSmallFwd) == (tid == 0))) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < kWarps; ++q) t += red[tid * kWarps + q];
    atomicAdd(tid == 0 ? p.loss_accum : p.dwdb + (tid - 1), t);
  }
  GE2E_SMALL_STAMP(5);
  if (p.stop == 4) break;
  if (PART == kSmallFwd) break;
  const bool vec_g = is_vec(p.dE_hat, D), vec_p = is_vec(p.part, D);
  {
    // thread <-> (float4 column c4 of 64, group of 4): dE_hat rows rg, rg + 4, ... = (wG) C_hat, then this speaker's
    // share (wG)^T E_hat of centroids kg, kg + 4, ...; a warp shares its group, so the w G entries are broadcasts
    const int d = (tid & 63) << 2, grp = tid >> 6;
    if (d < Dp) {
      float4 acc[R4];
#pragma unroll
      for (int q = 0; q < R4; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      // four centroids per step: the four w G entries of a row come as ONE broadcast 16-byte load (rows >= M are
      // zero; columns N..Np-1 of w G are never written, so the tail runs entry by entry)
      auto fma_row = [&](float4& a, float sgk, const float4& c) {
        a.x = fmaf(sgk, c.x, a.x); a.y = fmaf(sgk, c.y, a.y); a.z = fmaf(sgk, c.z, a.z); a.w = fmaf(sgk, c.w, a.w);
      };
      int k = 0;
      for (; k + 4 <= N; k += 4) {
        const float4 c0 = *reinterpret_cast<const float4*>(&sC[(size_t)(k + 0) * Ds + d]);
        const float4 c1 = *reinterpret_cast<const float4*>(&sC[(size_t)(k + 1) * Ds + d]);
        const float4 c2 = *reinterpret_cast<const float4*>(&sC[(size_t)(k + 2) * Ds + d]);
        const float4 c3 = *reinterpret_cast<const float4*>(&sC[(size_t)(k + 3) * Ds + d]);
#pragma unroll
        for (int q = 0; q < R4; ++q) {
          const float4 sg = *reinterpret_cast<const float4*>(&sG[(grp + 4 * q) * Np + k]);
          fma_row(acc[q], sg.x, c0); fma_row(acc[q], sg.y, c1); fma_row(acc[q], sg.z, c2); fma_row(acc[q], sg.w, c3);
        }
      }
      for (; k < N; ++k) {
        const float4 c = *reinterpret_cast<const float4*>(&sC[(size_t)k * Ds + d]);
#pragma unroll
        for (int q = 0; q < R4; ++q) fma_row(acc[q], sG[(grp + 4 * q) * Np + k], c);
      }
#pragma unroll
      for (int q = 0; q < R4; ++q) {
        const int i = grp + 4 * q;
        if (i < M) {
          st4(p.dE_hat + ((size_t)j * M + i) * D, d, D, vec_g, acc[q]);
          if (fast) *reinterpret_cast<float4*>(fU + (size_t)i * Dp + d) = acc[q];     // for the Jacobians (stage 3)
        }
      }
    }
    __syncthreads();                                   // the centroids are no longer needed: sC becomes the share tile
    GE2E_SMALL_STAMP(6);
    float* sP = sC;                                    // [N][Dp], contiguous (source of the bulk reduce-add)
    if (d < Dp) {
      float4 e[MR];
#pragma unroll
      for (int i = 0; i < MR; ++i) e[i] = *reinterpret_cast<const float4*>(&sEh[(size_t)i * Dp + d]);
      auto put_share = [&](int k, const float4& a) {
        if (dc_at_l2) *reinterpret_cast<float4*>(&sP[(size_t)k * Dp + d]) = a;
        else st4(p.part + ((size_t)j * N + k) * D, d, D, vec_p, a);
      };
      // centroids 4 grp + 16 t .. + 3: a row's four w G entries are one broadcast 16-byte load (rows >= M: w G and
      // e_hat are both zero -- no branch in the chain); the columns N..Np-1 of w G are never written: tail by entry
      int kb = 4 * grp;
      for (; kb + 4 <= N; kb += 16) {
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
        for (int i = 0; i < MR; ++i) {
          const float4 sg = *reinterpret_cast<const float4*>(&sG[i * Np + kb]);
          a0.x = fmaf(sg.x, e[i].x, a0.x); a0.y = fmaf(sg.x, e[i].y, a0.y); a0.z = fmaf(sg.x, e[i].z, a0.z); a0.w = fmaf(sg.x, e[i].w, a0.w);
          a1.x = fmaf(sg.y, e[i].x, a1.x); a1.y = fmaf(sg.y, e[i].y, a1.y); a1.z = fmaf(sg.y, e[i].z, a1.z); a1.w = fmaf(sg.y, e[i].w, a1.w);
          a2.x = fmaf(sg.z, e[i].x, a2.x); a2.y = fmaf(sg.z, e[i].y, a2.y); a2.z = fmaf(sg.z, e[i].z, a2.z); a2.w = fmaf(sg.z, e[i].w, a2.w);
          a3.x = fmaf(sg.w, e[i].x, a3.x); a3.y = fmaf(sg.w, e[i].y, a3.y); a3.z = fmaf(sg.w, e[i].z, a3.z); a3.w = fmaf(sg.w, e[i].w, a3.w);
        }
        put_share(kb, a0); put_share(kb + 1, a1); put_share(kb + 2, a2); put_share(kb + 3, a3);
      }
      for (int k = kb; k < N && k < kb + 4; ++k) {      // at most one group holds the N % 4 trailing centroids
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < MR; ++i) {
          const float sgk = sG[i * Np + k];
          a.x = fmaf(sgk, e[i].x, a.x); a.y = fmaf(sgk, e[i].y, a.y); a.z = fmaf(sgk, e[i].z, a.z); a.w = fmaf(sgk, e[i].w, a.w);
        }
        put_share(k, a);
      }
    }
    if (dc_at_l2) {
      ptx::fence_proxy_async_smem();                   // this thread's tile entries -> async proxy
      __syncthreads();
      GE2E_SMALL_STAMP(7);
      if (tid == 0) {
        asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;"
                     ::"l"(p.dC_hat), "r"(ptx::smem_u32(sP)), "r"(static_cast<uint32_t>((size_t)N * D * sizeof(float)))
                     : "memory");
        ptx::tma_store_commit();
      }
      if (fast) {
        // While the adds travel: everything of stage 3 that does not need the centroid gradient -- the two
        // normalisation Jacobians of e_hat and u_hat (same arithmetic as finalize_body) and the column sums of d u
        const bool act = hw < M;
        float eg = 0.f;
        if (act)
          for (int c4 = hl; c4 < ncol4; c4 += 16)
            eg += dot4(reinterpret_cast<const float4*>(fE + (size_t)hw * Dp)[c4],
                       reinterpret_cast<const float4*>(fU + (size_t)hw * Dp)[c4]);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) eg += __shfl_xor_sync(0xffffffffu, eg, o);
        if (act) {
          const float dd = diag_term(VARIANT, PART == kSmallBwd ? s_gr[hw] : g,
                                     VARIANT == GE2E_SOFTMAX ? s_aux[hw] : s_cd[hw], w, b, eps);
          const float3 rs = s_rsum[hw];
          const RowJacobian J = row_jacobian(row_norms(rs.x, rs.y, rs.z, inv_m1), eg, 1.f, dd, inv_m1);
          for (int c4 = hl; c4 < ncol4; c4 += 16) {
            const float4 e = reinterpret_cast<const float4*>(fE + (size_t)hw * Dp)[c4];
            const float4 sv = reinterpret_cast<const float4*>(fS)[c4];
            const float4 gv = reinterpret_cast<const float4*>(fU + (size_t)hw * Dp)[c4];
            const float ev[4] = {e.x, e.y, e.z, e.w}, ss[4] = {sv.x, sv.y, sv.z, sv.w}, gg[4] = {gv.x, gv.y, gv.z, gv.w};
            float de[4], du[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              de[t] = J.de(ev[t], ss[t] - ev[t], gg[t]);
              du[t] = J.du(ev[t], ss[t] - ev[t]);
            }
            // each slot is read and then overwritten by the same lane
            reinterpret_cast<float4*>(fU + (size_t)hw * Dp)[c4] = make_float4(du[0], du[1], du[2], du[3]);
            reinterpret_cast<float4*>(fE + (size_t)hw * Dp)[c4] = make_float4(de[0], de[1], de[2], de[3]);
          }
        }
        __syncthreads();          // d e, d u complete; the sums of the raw rows are no longer needed (c_mine)
        for (int d = tid; d < Dp; d += kThreads) {
          float sum = 0.f;
          for (int i = 0; i < M; ++i) sum += fU[(size_t)i * Dp + d];
          fS[d] = sum;
        }
      }
      // performed (not just read): the barrier arrival below publishes this CTA's adds
      if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
  }
  __syncthreads();
  if (!dc_at_l2) GE2E_SMALL_STAMP(7);
  if (p.stop == 5) break;
  if (p.cluster) { __syncthreads(); ptx::cluster_sync_all(); } else small_grid_barrier(p.ctr, (unsigned)(2 * N));
  GE2E_SMALL_STAMP(8);
  if (p.stop == 6) break;

  // ---- 3: centroid gradient of this speaker, then the Jacobians and the fan-out
  // (unaligned rows only: the block's threads split the N contributions into groups so that each thread has many
  // independent L2 loads in flight instead of a chain of N; the groups are then added in a fixed order)
  if (!dc_at_l2) {
    const int ncol4 = Dp >> 2;                               // <= 64 float4 columns
    const int ngrp = kThreads / ncol4;                       // >= 4 speaker groups
    const int col4 = tid % ncol4, grp = tid / ncol4;
    const int used = ngrp < N ? ngrp : N;
    float* sP = sC;                                          // [used][Dp]: the centroids are no longer needed
    __syncthreads();
    if (grp < used) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      const int col = col4 << 2;
      for (int j0 = grp; j0 < N; j0 += used * 8) {             // 8 L2 loads in flight, added in a fixed order
        float4 v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int jj = j0 + q * used;
          v[q] = (jj < N) ? ld4_cg(p.part + ((size_t)jj * N + j) * D, col, D, vec_p) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) { acc.x += v[q].x; acc.y += v[q].y; acc.z += v[q].z; acc.w += v[q].w; }
      }
      *reinterpret_cast<float4*>(&sP[(size_t)grp * Dp + col]) = acc;
    }
    __syncthreads();
    for (int d = tid; d < D; d += kThreads) {
      float sum = 0.f;
      for (int q = 0; q < used; ++q) sum += sP[(size_t)q * Dp + d];
      p.dC_hat[(size_t)j * D + d] = sum;
    }
  }
  __syncthreads();
  GE2E_SMALL_STAMP(9);
  if (p.stop == 7) break;
  if (fast) {
    const float dch = tid < D ? __ldcg(p.dC_hat + (size_t)j * D + tid) : 0.f;      // assembled at the L2 by all CTAs
    float prp = warp_sum(s_mine * dch);
    if (lane == 0) red[wid] = prp;
    __syncthreads();
    float pr = 0.f;
#pragma unroll
    for (int q = 0; q < kWarps; ++q) pr += red[q];
    if (tid < D) {
      const float2 k = centroid_jacobian(s_norm2, pr, inv_m);
      fB[tid] = dch * k.x - s_mine * k.y;     // dc_j / M
    }
    __syncthreads();
    for (int i = wid; i < M; i += kWarps) {           // fan-out of d c and of the leave-one-out centroids (s3:105-111)
      TD* dst = dE + phys_row(p.idx, (size_t)j * M + i) * D;
      for (int c4 = lane; c4 < ncol4; c4 += 32) {
        const float4 de = reinterpret_cast<const float4*>(fE + (size_t)i * Dp)[c4];
        const float4 du = reinterpret_cast<const float4*>(fU + (size_t)i * Dp)[c4];
        const float4 sd = reinterpret_cast<const float4*>(fS)[c4];
        const float4 bc = reinterpret_cast<const float4*>(fB)[c4];
        float4 o;
        o.x = de.x + bc.x + (sd.x - du.x) * inv_m1;
        o.y = de.y + bc.y + (sd.y - du.y) * inv_m1;
        o.z = de.z + bc.z + (sd.z - du.z) * inv_m1;
        o.w = de.w + bc.w + (sd.w - du.w) * inv_m1;
        st4v(dst + 4 * c4, o);
      }
    }
  } else if (PART == kSmallBwd) {
    finalize_body<true, TE, TD, true>(E, p.dE_hat, p.dC_hat, p.cos_diag, p.row_stat, p.row_aux, nullptr, j, M, D, Dp,
                                      w, b, 0.f, eps, VARIANT, dE, p.idx, sA, p.grad_rows);   // sA: stage_rows
  } else {
    finalize_body<true>(E, p.dE_hat, p.dC_hat, p.cos_diag, p.row_stat, p.row_aux, nullptr, j, M, D, Dp, w, b, g, eps,
                        VARIANT, dE, p.idx, sA);      // sA still holds the raw rows prep_body staged
  }
  } while (0);
  __syncthreads();
  GE2E_SMALL_STAMP(10);
  // last CTA out restores the workspace header (every CTA has left both barriers by the time it exits)
  if (tid == 0 && !p.cluster) {
    if (atomicAdd(p.ctr + 1, 1u) == (unsigned)(N - 1)) { atomicExch(p.ctr, 0u); atomicExch(p.ctr + 1, 0u); }
  }
}


size_t small_smem_bytes(int N, int M, int D) {
  const int Dp = (D + 3) & ~3, Np = (N + 3) & ~3, MR = (M + 3) & ~3;
  return ((size_t)(2 * M + 2 + MR) * Dp + (size_t)N * (Dp + 4) + (size_t)2 * MR * Np + (size_t)kWarps * MR * 32) *
         sizeof(float);
}

}  // namespace

// (contrast: the pipeline's backward is a two-non-zeros-per-row gather / scatter while the single kernel runs the
//  dense products; since the round-2 rewrite of the stages the single kernel still wins at cfg2: 19.7 vs 30.8 us)
bool small_step_preferred(int N, int M, int D, int variant) {
  return small_step_supported(N, M, D) && N <= (variant == GE2E_CONTRAST ? kSmallPickNContrast : kSmallPickN);
}

// The kernel's grid barriers need all N CTAs co-resident.  Counting one CTA per SM of the CURRENT device is
// conservative (small shapes would fit several) and also holds on a MIG slice, whose SM count is what the
// attribute reports; a device with fewer SMs than speakers takes the multi-kernel pipeline instead.
static int device_sm_count() {
  static int n[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  if (n[dev] == 0 && cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n[dev] = 0;
  return n[dev];
}

bool small_step_supported(int N, int M, int D) {
  return N >= 1 && N <= kSmallMaxN && M >= 2 && M <= kSmallMaxM && D >= 1 && D <= kSmallMaxD &&
         small_smem_bytes(N, M, D) <= 225 * 1024 && N <= device_sm_count();
}

size_t small_step_workspace_bytes(int N, int M, int D) {
  return small_step_supported(N, M, D) ? kSmallHeaderBytes + (size_t)N * N * D * sizeof(float) : 0;
}

int simt_small_step(int part, const void* E, int e_dt, const int32_t* row_index, int N, int M, int D, const float* w,
                    const float* b, float eps, int variant, const float* grad_out, const float* grad_rows, float* e_hat,
                    float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux, float* per_row,
                    float* loss_accum, float* dE_hat, float* dC_hat, float* dwdb, void* dE, int de_dt, void* workspace,
                    cudaStream_t st) {
  SmallParams p;
  p.E = E; p.idx = row_index; p.M = M; p.D = D; p.Dp = (D + 3) & ~3;
  p.w = w; p.b = b; p.eps = eps; p.grad_out = grad_out; p.grad_rows = grad_rows;
  p.e_hat = e_hat; p.c_hat = c_hat; p.cos_diag = cos_diag; p.row_stat = row_stat; p.row_kstar = row_kstar;
  p.row_aux = row_aux; p.per_row = per_row; p.loss_accum = loss_accum;
  p.dE_hat = dE_hat; p.dC_hat = dC_hat; p.dwdb = dwdb; p.dE = dE;
#ifdef GE2E_DEBUG_BUILD      // scripts/small_step_trace.py builds its own library with -DGE2E_DEBUG_BUILD
  static const int stop = [] { const char* e = getenv("GE2E_SMALL_STOP"); return e ? atoi(e) : 0; }();
  p.stop = part == kSmallWhole ? stop : 0;
#else
  p.stop = 0;
#endif
  p.ctr = reinterpret_cast<unsigned*>(workspace);
  p.part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + kSmallHeaderBytes);
  const size_t smem = small_smem_bytes(N, M, D);
  // N <= 8 (the portable cluster size): the N CTAs form one cluster
  p.cluster = N <= 8 ? 1 : 0;
  // the forward half stores no dE: one instantiation per E type
#define GE2E_SMALL_LAUNCH(V, R)                                                                   \
  do {                                                                                            \
    auto kern = part == kSmallFwd ? small_step_kernel<V, R, TE, float, kSmallFwd>                 \
              : part == kSmallBwd ? small_step_kernel<V, R, TE, TD, kSmallBwd>                    \
                                  : small_step_kernel<V, R, TE, TD, kSmallWhole>;                 \
    int rc = set_smem(kern, smem);                                                                \
    if (rc != GE2E_OK) return rc;                                                                 \
    cudaLaunchConfig_t cfg{};                                                                     \
    cfg.gridDim = dim3(N); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st; \
    cudaLaunchAttribute at[2];                                                                    \
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                \
    at[0].val.programmaticStreamSerializationAllowed = 1;                                         \
    at[1].id = cudaLaunchAttributeClusterDimension;                                               \
    at[1].val.clusterDim.x = N; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;           \
    cfg.attrs = at; cfg.numAttrs = p.cluster ? 2 : 1;                                             \
    GE2E_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p));                                             \
  } while (0)
  const int mr = (M + 3) & ~3;
  const int rc = with_e_de_types(e_dt, de_dt, [&](auto te, auto td) -> int {
    using TE = decltype(te);
    using TD = decltype(td);
    if (variant == GE2E_SOFTMAX) {
      if (mr == 4) GE2E_SMALL_LAUNCH(GE2E_SOFTMAX, 4); else if (mr == 8) GE2E_SMALL_LAUNCH(GE2E_SOFTMAX, 8);
      else if (mr == 12) GE2E_SMALL_LAUNCH(GE2E_SOFTMAX, 12); else GE2E_SMALL_LAUNCH(GE2E_SOFTMAX, 16);
    } else {
      if (mr == 4) GE2E_SMALL_LAUNCH(GE2E_CONTRAST, 4); else if (mr == 8) GE2E_SMALL_LAUNCH(GE2E_CONTRAST, 8);
      else if (mr == 12) GE2E_SMALL_LAUNCH(GE2E_CONTRAST, 12); else GE2E_SMALL_LAUNCH(GE2E_CONTRAST, 16);
    }
    return GE2E_OK;
  });
#undef GE2E_SMALL_LAUNCH
  if (rc != GE2E_OK) return rc;
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// The trainer's post-loss tail for the two loss parameters (s4_train_embed_model.py:202-203):
// clip_grad_norm_((w, b), max_norm) followed by the plain-SGD update, on the device, one thread.
// clip_grad_norm_ semantics: total = ||(dw, db)||_2, coef = min(1, max_norm / (total + 1e-6)),
// grads scaled in place (they stay visible to the caller), then p -= lr * grad.
__global__ void scale_bias_sgd_kernel(float* w, float* b, float* dw, float* db, float max_norm, float lr,
                                      float* total_norm) {
  pdl_wait();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float gw = *dw, gb = *db;
  const float total = sqrtf(gw * gw + gb * gb);
  const float coef = fminf(max_norm / (total + 1e-6f), 1.0f);
  const float cw = gw * coef, cb = gb * coef;
  *dw = cw;
  *db = cb;
  *w = *w - lr * cw;
  *b = *b - lr * cb;
  if (total_norm) *total_norm = total;
}

// Gradients of a step that ran with upstream gradient 1, scaled by the real one (the loss is linear in it):
// out = g * in, {dw, db}_out = g * {dw, db}_in.  One launch; the eager module path's backward.
// fp32 in; out is fp32 or a half type, each element rounded once after the scaling (so a small fp16 gradient times a
// loss scale keeps the digits it would lose if it were rounded first).
template <typename TO>
__global__ void __launch_bounds__(256)
scale_grads_kernel(const float* __restrict__ in, TO* __restrict__ out, long long n, const float* __restrict__ dwdb_in,
                   float* __restrict__ dwdb_out, const float* __restrict__ gp) {
  pdl_wait();
  const float g = __ldg(gp);
  if (blockIdx.x == 0 && threadIdx.x < 2) dwdb_out[threadIdx.x] = g * dwdb_in[threadIdx.x];
  const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if ((n & 3) == 0 && ((reinterpret_cast<uintptr_t>(in) & 15) | (reinterpret_cast<uintptr_t>(out) & (4 * sizeof(TO) - 1))) == 0) {
    const float4* i4 = reinterpret_cast<const float4*>(in);
    for (long long i = t0; i < (n >> 2); i += stride) {
      float4 v = __ldcs(i4 + i);
      v.x *= g; v.y *= g; v.z *= g; v.w *= g;
      if constexpr (std::is_same<TO, float>::value) __stcs(reinterpret_cast<float4*>(out) + i, v);
      else __stcs(reinterpret_cast<uint2*>(out) + i, narrow4<TO>(v));
    }
  } else {
    for (long long i = t0; i < n; i += stride) out[i] = from_f<TO>(g * in[i]);
  }
}

int simt_scale_grads(const float* in, void* out, int out_dt, long long n, const float* dwdb_in, float* dwdb_out,
                     const float* g, cudaStream_t st) {
  long long blocks = (n / 4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  with_e_type(out_dt, [&](auto to) -> int {
    using TO = decltype(to);
    launch_pdl(scale_grads_kernel<TO>, dim3((unsigned)blocks), dim3(256), 0, st, true, in, static_cast<TO*>(out), n,
               dwdb_in, dwdb_out, g);
    return GE2E_OK;
  });
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_scale_bias_sgd(float* w, float* b, float* dw, float* db, float max_norm, float lr, float* total_norm,
                        bool pdl, cudaStream_t st) {
  launch_pdl(scale_bias_sgd_kernel, dim3(1), dim3(32), 0, st, pdl, w, b, dw, db, max_norm, lr, total_norm);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// ---- EER sweep counts (s5_eval_model.py:57-89) ------------------------------------------------
// For every threshold t: how many entries of sim[N, M, N] exceed it, over the whole matrix and over
// the own-speaker entries sim[j, :, j].  One pass over the matrix: each value is binned by the number
// of (ascending) thresholds below it, bins are counted in shared-memory histograms (warp-aggregated:
// clustered embeddings put most of a warp into the same bin), and the last block turns the histograms
// into "accepted at threshold t" = sum of the bins above t.  Integer work, bit-exact by construction.
// Up to kEerPrivT thresholds (the reference uses 50) every lane owns a private column of its warp's
// histogram (bank = lane: plain conflict-free read-modify-write, no atomics); beyond that the warps of a
// block share one histogram through warp-aggregated shared-memory atomics.
constexpr int kEerMaxT = 1024;
constexpr int kEerThreads = 256;
constexpr int kEerPrivT = 64;
constexpr int kEerPrivThreads = 512;   // few large blocks: the per-block fold ends in same-address global atomics

__device__ __forceinline__ int eer_bin(float v, const float* thr, int T) {
  int lo = 0, hi = T;                      // number of thresholds with v > thr  (NaN -> 0)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (v > thr[mid]) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// The same count, reached from a linear guess between the first and the last threshold and two
// verifying compares (thr[g-1] < v, !(thr[g] < v)); the guess only ever saves the search -- a wrong
// one (unevenly spaced thresholds, a value exactly on a threshold) falls back to it.  The reference's
// thresholds are an even grid (s5:57), for which the guess is right except on ties.
__device__ __forceinline__ int eer_bin_guess(float v, const float* thr, int T, float lo, float inv) {
  const float f = (v - lo) * inv;
  const int g = (f >= 0.f) ? ((f < (float)T) ? (int)f + 1 : T) : 0;      // NaN -> 0
  const bool ok_lo = (g == 0) || (v > thr[g - 1]);
  const bool ok_hi = (g == T) || !(v > thr[g]);
  if (ok_lo && ok_hi) return g;
  return eer_bin(v, thr, T);
}

__device__ __forceinline__ void eer_count(unsigned* hist, int bin, bool on) {
  const unsigned act = __ballot_sync(0xffffffffu, on);
  if (!on) return;
  const unsigned peers = __match_any_sync(act, bin);
  if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&hist[bin], (unsigned)__popc(peers));
}

// accepted at threshold t = values with more than t thresholds below them = sum of bins t+1 .. T
// (the whole last block fetches the two histograms into shared memory first: a single thread walking them
// in global memory is a chain of T dependent L2 round trips, ~17 us at T = 50)
__device__ __forceinline__ void eer_finish(unsigned long long* hist_g, int T, long long* accept_all, long long* accept_own,
                                           unsigned long long* s_h /* shared, 2 (T + 1) entries */) {
  const volatile unsigned long long* h = hist_g;
  for (int i = threadIdx.x; i < 2 * (T + 1); i += blockDim.x) s_h[i] = h[i];
  __syncthreads();
  if (threadIdx.x < 2) {
    const unsigned long long* hs = s_h + threadIdx.x * (T + 1);
    long long* out = threadIdx.x == 0 ? accept_all : accept_own;
    long long run = 0;
    for (int t = T - 1; t >= 0; --t) {
      run += (long long)hs[t + 1];
      out[t] = run;
    }
  }
}

__global__ void __launch_bounds__(kEerPrivThreads)
threshold_counts_private_kernel(const float* __restrict__ sim, long long rows, int N, int M,
                                const float* __restrict__ thr_g, int T, unsigned long long* __restrict__ hist_g,
                                long long* __restrict__ accept_all, long long* __restrict__ accept_own) {
  extern __shared__ __align__(16) unsigned eer_smem[];
  constexpr int kWarps = kEerPrivThreads / 32;
  float* thr = reinterpret_cast<float*>(eer_smem);            // [T]
  unsigned* h_own = eer_smem + T;                              // [T + 1]
  unsigned* priv = h_own + (T + 1);                            // [kWarps][T + 1][32]
  __shared__ bool last;
  for (int i = threadIdx.x; i < T; i += blockDim.x) thr[i] = thr_g[i];
  for (int i = threadIdx.x; i < (T + 1) * (1 + kWarps * 32); i += blockDim.x) h_own[i] = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned* mine = priv + (size_t)warp * (T + 1) * 32 + lane;
  const float g_lo = thr[0];
  const float g_span = thr[T - 1] - thr[0];
  const float g_inv = g_span > 0.f ? (float)(T - 1) / g_span : 0.f;
  const long long nwarps = (long long)gridDim.x * kWarps;
  for (long long row = (long long)blockIdx.x * kWarps + warp; row < rows; row += nwarps) {
    const int j = (int)(row / M);
    const float* src = sim + row * N;
    int k = lane;
    // eight loads and searches in flight per lane (the kernel is latency-bound otherwise)
    for (; k + 224 < N; k += 256) {
      float v[8];
      int bn[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = __ldg(src + k + 32 * q);
#pragma unroll
      for (int q = 0; q < 8; ++q) bn[q] = eer_bin_guess(v[q], thr, T, g_lo, g_inv);
#pragma unroll
      for (int q = 0; q < 8; ++q) mine[bn[q] * 32] += 1u;
      const int dj = j - k;
      if (dj >= 0 && dj < 256 && (dj & 31) == 0) {
        int b = bn[0];
#pragma unroll
        for (int q = 1; q < 8; ++q) b = (dj == 32 * q) ? bn[q] : b;
        atomicAdd(&h_own[b], 1u);
      }
    }
    for (; k < N; k += 32) {
      const int b = eer_bin_guess(__ldg(src + k), thr, T, g_lo, g_inv);
      mine[b * 32] += 1u;
      if (k == j) atomicAdd(&h_own[b], 1u);
    }
  }
  __syncthreads();
  // fold the private columns: thread `bin` walks its row of 32 columns starting at a different bank
  for (int bin = threadIdx.x; bin <= T; bin += blockDim.x) {
    unsigned long long sum = 0;
    for (int w = 0; w < kWarps; ++w)
      for (int i = 0; i < 32; ++i) sum += priv[((size_t)w * (T + 1) + bin) * 32 + ((i + bin) & 31)];
    if (sum) atomicAdd(&hist_g[bin], sum);
    if (h_own[bin]) atomicAdd(&hist_g[T + 1 + bin], (unsigned long long)h_own[bin]);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&hist_g[2 * (T + 1)], 1ull) == (unsigned long long)(gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  __syncthreads();
  eer_finish(hist_g, T, accept_all, accept_own, reinterpret_cast<unsigned long long*>(eer_smem));
}

__global__ void __launch_bounds__(kEerThreads)
threshold_counts_kernel(const float* __restrict__ sim, long long total, int N, int M, const float* __restrict__ thr_g,
                        int T, unsigned long long* __restrict__ hist_g /* [2][T+1] + ticket */,
                        long long* __restrict__ accept_all, long long* __restrict__ accept_own) {
  extern __shared__ __align__(16) unsigned eer_smem[];
  float* thr = reinterpret_cast<float*>(eer_smem);            // [T]
  unsigned* h_all = eer_smem + T;                              // [T + 1]
  unsigned* h_own = h_all + (T + 1);                           // [T + 1]
  __shared__ bool last;
  for (int i = threadIdx.x; i < T; i += blockDim.x) thr[i] = thr_g[i];
  for (int i = threadIdx.x; i < 2 * (T + 1); i += blockDim.x) h_all[i] = 0u;
  __syncthreads();
  // one warp per row sim[j, i, :] (whole warps stay in the loops together: ballot / match need every
  // lane, so both bounds are warp-uniform); the own-speaker entry of the row is k == j
  const int lane = threadIdx.x & 31;
  const long long rows = total / N;
  const long long nwarps = (long long)gridDim.x * (kEerThreads / 32);
  for (long long row = (long long)blockIdx.x * (kEerThreads / 32) + (threadIdx.x >> 5); row < rows; row += nwarps) {
    const int j = (int)(row / M);
    const float* src = sim + row * N;
    for (int k0 = 0; k0 < N; k0 += 32) {
      const int k = k0 + lane;
      const bool on = k < N;
      const float v = on ? __ldg(src + k) : 0.f;
      const int bin = on ? eer_bin(v, thr, T) : 0;
      eer_count(h_all, bin, on);
      eer_count(h_own, bin, on && k == j);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * (T + 1); i += blockDim.x)
    if (h_all[i]) atomicAdd(&hist_g[i], (unsigned long long)h_all[i]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&hist_g[2 * (T + 1)], 1ull) == (unsigned long long)(gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  __syncthreads();
  eer_finish(hist_g, T, accept_all, accept_own, reinterpret_cast<unsigned long long*>(eer_smem));
}

int simt_threshold_counts(const float* sim, int N, int M, const float* thresholds, int T, long long* accept_all,
                          long long* accept_own, void* scratch, cudaStream_t st) {
  if (T < 1 || T > kEerMaxT) return GE2E_ERR_UNSUPPORTED;
  const long long total = (long long)N * M * N;
  const size_t scratch_bytes = (size_t)(2 * (T + 1) + 1) * sizeof(unsigned long long);
  if (cudaMemsetAsync(scratch, 0, scratch_bytes, st) != cudaSuccess) return GE2E_ERR_LAUNCH;
  const long long rows = (long long)N * M;                     // one warp per row sim[j, i, :]
  constexpr int kSms = 148;
  unsigned long long* hist = reinterpret_cast<unsigned long long*>(scratch);
  if (T <= kEerPrivT) {
    constexpr int kWarps = kEerPrivThreads / 32;
    const size_t smem = (size_t)(T + (T + 1) * (1 + kWarps * 32)) * sizeof(unsigned);      // <= 134 KB
    int rc = set_smem(threshold_counts_private_kernel, smem);
    if (rc != GE2E_OK) return rc;
    long long blocks = (rows + kWarps - 1) / kWarps;
    const long long cap = (long long)kSms * (smem <= 110 * 1024 ? 2 : 1);   // resident blocks per SM by shared memory
    if (blocks > cap) blocks = cap;
    threshold_counts_private_kernel<<<(unsigned)blocks, kEerPrivThreads, smem, st>>>(sim, rows, N, M, thresholds, T, hist,
                                                                                     accept_all, accept_own);
  } else {
    long long blocks = (rows + kEerThreads / 32 - 1) / (kEerThreads / 32);
    const long long cap = (long long)kSms * 8;                 // 8 resident blocks of 256 threads per SM
    if (blocks > cap) blocks = cap;
    // the last block re-uses the dynamic shared memory for 2 (T + 1) 64-bit histogram entries
    const size_t smem = std::max((size_t)(T + 2 * (T + 1)) * sizeof(unsigned), (size_t)2 * (T + 1) * sizeof(unsigned long long));
    threshold_counts_kernel<<<(unsigned)blocks, kEerThreads, smem, st>>>(sim, total, N, M, thresholds, T, hist, accept_all,
                                                                         accept_own);
  }
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// ---- batch assembly from a device-resident spectrogram bank (s1_dataset_loader.py:59-77) -------
// A cropped utterance [crop_len, mels] is ONE contiguous span of the speaker's [utts, frames, mels]
// array, so assembling the model's input batch (collate + reshape + the trainer's row permutation,
// s4:176-186) is `rows` contiguous copies: out[r, :] = bank[src_off[r] : src_off[r] + span].
// Pure HBM copy work: a block copies one chunk of one span, 16-byte vectors, four loads in flight per
// thread; spans or offsets that are not 16-byte multiples take the scalar kernel.
constexpr int kGatherThreads = 256;
constexpr int kGatherChunk = kGatherThreads * 4 * 4;          // floats per block: 4 float4 per thread

__global__ void __launch_bounds__(kGatherThreads)
gather_spans_vec_kernel(const float* __restrict__ bank, const long long* __restrict__ src_off, long long span,
                        int chunks, float* __restrict__ out) {
  const int row = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const long long off = __ldg(src_off + row);
  const float4* src = reinterpret_cast<const float4*>(bank + off);
  float4* dst = reinterpret_cast<float4*>(out + (long long)row * span);
  const long long n4 = span >> 2;
  const long long base = (long long)chunk * (kGatherChunk / 4) + threadIdx.x;
  float4 v[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const long long i = base + (long long)q * kGatherThreads;
    if (i < n4) v[q] = __ldcs(src + i);                        // read once: do not keep the bank in L2
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const long long i = base + (long long)q * kGatherThreads;
    if (i < n4) dst[i] = v[q];
  }
}

__global__ void __launch_bounds__(kGatherThreads)
gather_spans_scalar_kernel(const float* __restrict__ bank, const long long* __restrict__ src_off, long long span,
                           int chunks, float* __restrict__ out) {
  const int row = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const float* src = bank + __ldg(src_off + row);
  float* dst = out + (long long)row * span;
  const long long lo = (long long)chunk * kGatherChunk;
  const long long hi = lo + kGatherChunk < span ? lo + kGatherChunk : span;
  for (long long i = lo + threadIdx.x; i < hi; i += kGatherThreads) dst[i] = __ldg(src + i);
}

int simt_gather_spans(const float* bank, const long long* src_off, int rows, long long span, bool vec_ok, float* out,
                      cudaStream_t st) {
  const long long chunks = (span + kGatherChunk - 1) / kGatherChunk;
  const long long blocks = chunks * rows;
  if (blocks > 0x7fffffffLL) return GE2E_ERR_UNSUPPORTED;
  if (vec_ok) gather_spans_vec_kernel<<<(unsigned)blocks, kGatherThreads, 0, st>>>(bank, src_off, span, (int)chunks, out);
  else gather_spans_scalar_kernel<<<(unsigned)blocks, kGatherThreads, 0, st>>>(bank, src_off, span, (int)chunks, out);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// ------------------------------------------------------------------------------------------
// Speaker-sharded step over peer memory (NVLink / NVSwitch): the all-gather of the normalised centroids as
// plain stores.  Every rank copies ITS slice of c_hat (1 MB at config 4 on 8 ranks) into the same slice of
// every peer's c_hat_all and clears its own dC_local, which the peers' step kernels then add into.
// ------------------------------------------------------------------------------------------
namespace {
struct PeerDst { float4* p[GE2E_MAX_PEERS]; };

template <bool MULTICAST>
__global__ void __launch_bounds__(256)
peer_publish_kernel(const float4* __restrict__ src, PeerDst dst, int n_dst, long long n4, float4* __restrict__ zero,
                    long long zero_n4) {
  pdl_wait();        // src is written by the preceding kernel
  pdl_trigger();
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = src[i];
    if (MULTICAST) {
      // dst.p[0] is a multicast address of the NVSwitch domain: ONE store leaves this GPU, the switch
      // replicates it into every rank's copy of the buffer (this rank's own included)
      asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst.p[0] + i), "f"(v.x),
                   "f"(v.y), "f"(v.z), "f"(v.w)
                   : "memory");
    } else {
#pragma unroll
      for (int r = 0; r < GE2E_MAX_PEERS; ++r)
        if (r < n_dst) dst.p[r][i] = v;
    }
  }
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < zero_n4; i += stride)
    zero[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}
}  // namespace

int simt_peer_publish(const float* src, float* const* dst, int n_dst, bool multicast, long long n_floats, float* zero,
                      long long zero_floats, cudaStream_t st) {
  PeerDst d{};
  for (int r = 0; r < n_dst; ++r) d.p[r] = reinterpret_cast<float4*>(dst[r]);
  const long long n4 = n_floats / 4, z4 = zero_floats / 4;
  const int grid = static_cast<int>(std::min<long long>(148 * 2, std::max<long long>(1, (std::max(n4, z4) + 255) / 256)));
  if (multicast)
    GE2E_CUDA_TRY(launch_pdl(peer_publish_kernel<true>, dim3(grid), dim3(256), 0, st, true,
                             reinterpret_cast<const float4*>(src), d, n_dst, n4, reinterpret_cast<float4*>(zero), z4));
  else
    GE2E_CUDA_TRY(launch_pdl(peer_publish_kernel<false>, dim3(grid), dim3(256), 0, st, true,
                             reinterpret_cast<const float4*>(src), d, n_dst, n4, reinterpret_cast<float4*>(zero), z4));
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_centroids(const float* E, int N, int M, int D, float* C, cudaStream_t st) {
  centroids_kernel<<<N, 128, 0, st>>>(E, M, D, C);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_utterance_centroids(const float* E, int N, int M, int D, float* Uc, cudaStream_t st) {
  utt_centroids_kernel<<<N, 128, 0, st>>>(E, M, D, Uc);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_normalize_rows(const float* X, int rows, int D, float* Y, cudaStream_t st) {
  normalize_rows_kernel<<<(rows + kWarps - 1) / kWarps, kThreads, 0, st>>>(X, rows, D, Y);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

int simt_calc_loss(const float* S, int N, int M, float eps, int variant, float* loss, float* per_row,
                   cudaStream_t st) {
  GE2E_CUDA_TRY(cudaMemsetAsync(loss, 0, sizeof(float), st));
  calc_loss_kernel<<<(N * M + kWarps - 1) / kWarps, kThreads, 0, st>>>(S, N, M, eps, variant, loss, per_row);
  GE2E_LAUNCHED();
  return GE2E_OK;
}

}  // namespace ge2e
