// Fused BatchNorm(train) + residual add + sign/pack around the binary conv (SURVEY.md §8f rank 1: "the
// step either side of the conv").  The binary conv writes y; these kernels replace the cuDNN BN
// forward/backward, the ATen residual adds and the separate act_pack / grad_amax / grad_pack passes:
//
//   forward : bn_stats (1 read of y)  ->  bn_finalize ([C] math + running stats)
//             bn_apply_add_pack: z = y*a[c] + b[c] (+ residual)  [+ sign bits, STE mask bits and the +-1
//             16-bit copy of z, i.e. the NEXT conv's act_pack, in the same pass]
//   backward: bn_bwd_reduce (1 read of gz,y: sum gz, sum gz*yhat, max|gz| per channel)
//             bn_bwd_bound  ([C] math: dgamma, dbeta, per-channel constants, FP16S scale from a bound)
//             bn_bwd_pack   (1 read of gz,y -> gys = 16-bit operand of dgrad_tc / wgrad_tc; the fp32
//                            conv-output gradient is never materialised)
// Per element: forward 4 + 12(+2.25) bytes instead of 12 (BN) + 12 (add) + 6.25 (pack);
//              backward 8 + 10 bytes instead of ~20 (BN bwd) + 4 (amax) + 6 (pack).
// All tensors fp32 NHWC [n_pix][C], C % 4 == 0 (packing: C % 32 == 0).
#include <cuda_fp16.h>

#include "common.cuh"

namespace bdbnn {

constexpr int kBnThreads = 256;

__device__ __forceinline__ uint32_t bn_pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t bn_pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bn_bf16_round(float v) {
  return __uint_as_float(bn_pack_bf16x2(0.f, v) & 0xffff0000u);
}

// y operand of the fused units: fp32 (y itself) or the exact int16 accumulator y_int with y = alpha[c]*y_int
// (bdbnn_binconv_fwd_tc_i16).  The loaders return y_int as floats for I16 — callers fold alpha into their
// per-channel constants, which is exact in the same sense (one fp32 multiply either way).
template <bool I16>
__device__ __forceinline__ float4 load_y4(const void* __restrict__ y, int64_t i) {
  if (I16) {
    const uint2 r = __ldcs(reinterpret_cast<const uint2*>(y) + i);
    return make_float4(float(int16_t(r.x & 0xffffu)), float(int16_t(r.x >> 16)), float(int16_t(r.y & 0xffffu)),
                       float(int16_t(r.y >> 16)));
  }
  return __ldcs(reinterpret_cast<const float4*>(y) + i);
}

// Per-channel (sum a, sum b, max c) over pixels; thread = one float4 channel group, strided over pixels.
// Block partials go through shared-memory atomics, then one double atomicAdd per channel per block.  The threads'
// fp32 partials meet in fp64 (exact while they span fewer than ~29 binary orders of magnitude, otherwise rounded in
// the last fp64 bits), so the arrival order of the atomics almost never reaches the fp32 statistics.
template <bool BWD, bool I16 = false>
__global__ void __launch_bounds__(kBnThreads)
bn_reduce_kernel(const float4* __restrict__ p0, const void* __restrict__ p1, const float* __restrict__ mean,
                 const float* __restrict__ invstd, int64_t n_pix, int C4, double* __restrict__ sums,
                 uint32_t* __restrict__ maxbits, const float* __restrict__ alpha = nullptr) {
  extern __shared__ double sh[];              // [2][C] sums, then [C] max bits (bn_reduce_smem)
  const int C = C4 * 4;
  uint32_t* shm = reinterpret_cast<uint32_t*>(sh + 2 * C);   // non-negative floats order like uints
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) sh[i] = 0.0;
  for (int i = threadIdx.x; i < C; i += blockDim.x) shm[i] = 0u;
  __syncthreads();
  const int64_t gtid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;   // multiple of C4 (host guarantees)
  const int c4 = int(gtid % C4);
  const int64_t p_step = nthreads / C4;
  float4 mu = make_float4(0, 0, 0, 0), is = make_float4(1, 1, 1, 1);
  if (BWD) {
    mu = *reinterpret_cast<const float4*>(mean + c4 * 4);
    is = *reinterpret_cast<const float4*>(invstd + c4 * 4);
    if (I16) {     // yhat = (alpha*yi - mean)*invstd = (yi - mean/alpha) * (alpha*invstd); alpha == 0 -> yhat = -mean*invstd
      const float4 al = *reinterpret_cast<const float4*>(alpha + c4 * 4);
      // keep the exact form: yhat = yi*(alpha*is) - mean*is, expressed through (v - mu')*is' with v = yi
      mu = make_float4(mu.x * is.x, mu.y * is.y, mu.z * is.z, mu.w * is.w);           // mean*invstd
      is = make_float4(al.x * is.x, al.y * is.y, al.z * is.z, al.w * is.w);           // alpha*invstd
    }
  }
  float4 sa = make_float4(0, 0, 0, 0), sb = sa, mx = sa;
#pragma unroll 8
  for (int64_t p = gtid / C4; p < n_pix; p += p_step) {
    const float4 u = __ldcs(p0 + p * C4 + c4);
    if (BWD) {   // u = gz, v = y:  a = gz, b = gz * yhat, c = |gz|
      const float4 v = load_y4<I16>(p1, p * C4 + c4);
      sa.x += u.x; sa.y += u.y; sa.z += u.z; sa.w += u.w;
      if (I16) {
        sb.x += u.x * fmaf(v.x, is.x, -mu.x); sb.y += u.y * fmaf(v.y, is.y, -mu.y);
        sb.z += u.z * fmaf(v.z, is.z, -mu.z); sb.w += u.w * fmaf(v.w, is.w, -mu.w);
      } else {
        sb.x += u.x * ((v.x - mu.x) * is.x); sb.y += u.y * ((v.y - mu.y) * is.y);
        sb.z += u.z * ((v.z - mu.z) * is.z); sb.w += u.w * ((v.w - mu.w) * is.w);
      }
    } else {     // u = y:  a = y, b = y*y, c = |y|
      sa.x += u.x; sa.y += u.y; sa.z += u.z; sa.w += u.w;
      sb.x += u.x * u.x; sb.y += u.y * u.y; sb.z += u.z * u.z; sb.w += u.w * u.w;
    }
    mx.x = fmaxf(mx.x, fabsf(u.x)); mx.y = fmaxf(mx.y, fabsf(u.y));
    mx.z = fmaxf(mx.z, fabsf(u.z)); mx.w = fmaxf(mx.w, fabsf(u.w));
  }
  const int c = c4 * 4;
  atomicAdd(&sh[c + 0], double(sa.x)); atomicAdd(&sh[c + 1], double(sa.y));
  atomicAdd(&sh[c + 2], double(sa.z)); atomicAdd(&sh[c + 3], double(sa.w));
  atomicAdd(&sh[C + c + 0], double(sb.x)); atomicAdd(&sh[C + c + 1], double(sb.y));
  atomicAdd(&sh[C + c + 2], double(sb.z)); atomicAdd(&sh[C + c + 3], double(sb.w));
  atomicMax(&shm[c + 0], __float_as_uint(mx.x)); atomicMax(&shm[c + 1], __float_as_uint(mx.y));
  atomicMax(&shm[c + 2], __float_as_uint(mx.z)); atomicMax(&shm[c + 3], __float_as_uint(mx.w));
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    atomicAdd(sums + i, sh[i]);
    atomicAdd(sums + C + i, sh[C + i]);
    atomicMax(maxbits + i, shm[i]);
  }
}

// Dynamic shared memory of bn_reduce_kernel: [2][C] fp64 sums + [C] max bits; above the default 48 KB (C > 2457)
// the kernel has to opt in first.
static size_t bn_reduce_smem(int C) { return size_t(C) * (2 * sizeof(double) + sizeof(uint32_t)); }
template <typename Kernel>
static cudaError_t bn_reduce_allow(Kernel kernel, int C) {
  return bn_reduce_smem(C) > 48 * 1024
             ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bn_reduce_smem(C)))
             : cudaSuccess;
}

// [C] math of the forward: mean, invstd, a = gamma*invstd, b = beta - mean*a, running statistics
// (torch.nn.BatchNorm2d: biased variance for normalisation, unbiased for running_var).
__global__ void bn_finalize_kernel(const double* __restrict__ sums, int64_t n_pix, int C, float eps,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ mean, float* __restrict__ invstd, float* __restrict__ a,
                                   float* __restrict__ b, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float momentum,
                                   const float* __restrict__ alpha_i16 = nullptr) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double n = double(n_pix);
  const double m = sums[c] / n;
  double var = sums[C + c] / n - m * m;
  if (var < 0.0) var = 0.0;
  const float is = float(1.0 / sqrt(var + double(eps)));
  const float mf = float(m);
  mean[c] = mf;
  invstd[c] = is;
  const float av = gamma[c] * is;
  a[c] = alpha_i16 != nullptr ? av * alpha_i16[c] : av;     // int16 operand: z = y_int * (a*alpha) + b
  b[c] = beta[c] - mf * av;
  if (running_mean != nullptr) {
    const double unb = n > 1.0 ? var * n / (n - 1.0) : var;
    running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * mf;
    running_var[c] = (1.0f - momentum) * running_var[c] + momentum * float(unb);
  }
}

// z = y*a + b (+ residual); optionally the sign / STE-mask bits and the +-1 16-bit copy of z.
template <bool PACK, bool I16 = false, int U = 4>
__global__ void __launch_bounds__(kBnThreads)
bn_apply_add_pack_kernel(const void* __restrict__ y, const float4* __restrict__ res,
                         const float* __restrict__ a, const float* __restrict__ b, int64_t n4, int C4,
                         float4* __restrict__ z, uint32_t* __restrict__ sign_bits,
                         uint32_t* __restrict__ mask_bits, uint2* __restrict__ xb4, uint32_t* __restrict__ xb8,
                         uint32_t one16) {
  const int lane = threadIdx.x & 31;
  const uint32_t group_mask = 0xffu << (lane & 24);
  const int sh = (lane & 7) * 4;
  const uint32_t pos = one16, neg = one16 | 0x8000u;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;       // multiple of C4 (host guarantees)
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c4 = int(i % C4);                                     // constant per thread
  const float4 av = *reinterpret_cast<const float4*>(a + c4 * 4);
  const float4 bv = *reinterpret_cast<const float4*>(b + c4 * 4);
  auto emit = [&](int64_t i, const float4 v, const float4 r) {
    float4 o = make_float4(fmaf(v.x, av.x, bv.x), fmaf(v.y, av.y, bv.y), fmaf(v.z, av.z, bv.z),
                           fmaf(v.w, av.w, bv.w));
    o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    // z (4 B/element, re-read only after the next conv has run) is stored evict-first so that the next conv's
    // operands written below (xb / xb8, 1-2 B/element) have a chance to stay in the 126 MB L2
    __stcs(z + i, o);
    if (PACK) {
      const uint32_t s0 = o.x >= 0.0f, s1 = o.y >= 0.0f, s2 = o.z >= 0.0f, s3 = o.w >= 0.0f;
      const uint32_t m0 = fabsf(o.x) <= 1.0f, m1 = fabsf(o.y) <= 1.0f, m2 = fabsf(o.z) <= 1.0f,
                     m3 = fabsf(o.w) <= 1.0f;
      const uint32_t sw = __reduce_or_sync(group_mask, (s0 | (s1 << 1) | (s2 << 2) | (s3 << 3)) << sh);
      const uint32_t mw = __reduce_or_sync(group_mask, (m0 | (m1 << 1) | (m2 << 2) | (m3 << 3)) << sh);
      if ((lane & 7) == 0) {
        sign_bits[i >> 3] = sw;
        mask_bits[i >> 3] = mw;
      }
      uint2 q;
      q.x = (s0 ? pos : neg) | ((s1 ? pos : neg) << 16);
      q.y = (s2 ? pos : neg) | ((s3 ? pos : neg) << 16);
      xb4[i] = q;
      if (xb8 != nullptr)   // e4m3 +-1 bytes for the fp8 forward of the next conv
        xb8[i] = 0x38383838u | ((s0 ? 0u : 0x80u) | (s1 ? 0u : 0x8000u) | (s2 ? 0u : 0x800000u) | (s3 ? 0u : 0x80000000u));
    }
  };
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  // two elements per thread and iteration: all four loads are issued before the first dependent instruction
  // (whole 8-lane pack groups take the same branch: n4 and nthreads are multiples of 8)
  for (; i + (U - 1) * nthreads < n4; i += U * nthreads) {
    float4 v[U], r[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = load_y4<I16>(y, i + u * nthreads);       // I16: `a` already carries alpha
#pragma unroll
    for (int u = 0; u < U; ++u) r[u] = res != nullptr ? __ldcs(res + i + u * nthreads) : zero4;
#pragma unroll
    for (int u = 0; u < U; ++u) emit(i + u * nthreads, v[u], r[u]);
  }
  for (; i < n4; i += nthreads) emit(i, load_y4<I16>(y, i), res != nullptr ? __ldcs(res + i) : zero4);
}

// [C] math of the backward.  consts[c] = {m1, m2*invstd, mean, a*gscale}; gy*gscale = (gz - m1 -
// (y-mean)*m2*invstd) * a*gscale.  FP16S scale from the bound
//   |gy*gscale| <= |a*gscale| * (max|gz| + |m1| + (max|y| + |mean|)*invstd*|m2|).
__global__ void bn_bwd_bound_kernel(const double* __restrict__ sums, const uint32_t* __restrict__ gmax_bits,
                                    const uint32_t* __restrict__ ymax_bits, int64_t n_pix, int C,
                                    const float* __restrict__ mean, const float* __restrict__ invstd,
                                    const float* __restrict__ gamma, const float* __restrict__ gscale,
                                    float4* __restrict__ consts, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta, uint32_t* __restrict__ amax_bits,
                                    float gz_mult = 1.0f, const float* __restrict__ alpha_i16 = nullptr) {
  __shared__ float red[32];
  float bound = 0.f;
  const double n = double(n_pix);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float s1 = float(sums[c]), s2 = float(sums[C + c]);
    dbeta[c] = s1;
    dgamma[c] = s2;
    const float m1 = float(sums[c] / n), m2 = float(sums[C + c] / n);
    const float is = invstd[c], mu = mean[c];
    const float A = gamma[c] * is * gscale[c];
    // pack kernel: (gz - k.x - (v - k.z)*k.y) * k.w with v = y; for the int16 operand v = y_int, so
    // (y - mu)*m2*is = (y_int - mu/alpha) * (alpha*m2*is)   (alpha == 0: y == 0 everywhere, term = -mu*m2*is)
    if (alpha_i16 != nullptr) {
      const float al = alpha_i16[c];
      if (al != 0.f) consts[c] = make_float4(m1, al * m2 * is, mu / al, A);
      else           consts[c] = make_float4(m1 - mu * m2 * is, 0.f, 0.f, A);
    } else {
      consts[c] = make_float4(m1, m2 * is, mu, A);
    }
    const float ymax = __uint_as_float(ymax_bits[c]), gmax = __uint_as_float(gmax_bits[c]);
    // gz_mult: how many gradient values can land on one position (pooled stem: windows per pixel)
    bound = fmaxf(bound, fabsf(A) * (gz_mult * gmax + fabsf(m1) + (ymax + fabsf(mu)) * is * fabsf(m2)));
  }
  bound = warp_max(bound);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = bound;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int i = 0; i < int(blockDim.x >> 5); ++i) m = fmaxf(m, red[i]);
    *amax_bits = __float_as_uint(m);
  }
}

// gys = 16-bit operand of the conv backward, straight from gz and y.
template <int MODE, bool I16 = false, int U = 4>
__global__ void __launch_bounds__(kBnThreads)
bn_bwd_pack_kernel(const float4* __restrict__ gz, const void* __restrict__ y, const float4* __restrict__ consts,
                   const uint32_t* __restrict__ amax_bits, int64_t n4, int C4, uint16_t* __restrict__ out) {
  constexpr int HALVES = MODE == 2 ? 2 : 1;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;       // multiple of C4
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c4 = int(i % C4);
  const float up = MODE == 3 ? amax_pow2_scale(*amax_bits, false) : 1.0f;
  const float4 k0 = consts[c4 * 4 + 0], k1 = consts[c4 * 4 + 1], k2 = consts[c4 * 4 + 2], k3 = consts[c4 * 4 + 3];
  const int C = C4 * 4;
  int64_t pix = i / C4;
  const int64_t pix_step = nthreads / C4;
  auto emit = [&](int64_t pix, const float4 g, const float4 v) {
    const float a0 = (g.x - k0.x - (v.x - k0.z) * k0.y) * k0.w * up;
    const float a1 = (g.y - k1.x - (v.y - k1.z) * k1.y) * k1.w * up;
    const float a2 = (g.z - k2.x - (v.z - k2.z) * k2.y) * k2.w * up;
    const float a3 = (g.w - k3.x - (v.w - k3.z) * k3.y) * k3.w * up;
    uint2 r;
    if (MODE == 3) {
      r.x = bn_pack_f16x2(a0, a1);
      r.y = bn_pack_f16x2(a2, a3);
    } else {
      r.x = bn_pack_bf16x2(a0, a1);
      r.y = bn_pack_bf16x2(a2, a3);
    }
    uint16_t* dst = out + pix * (int64_t(HALVES) * C) + c4 * 4;
    *reinterpret_cast<uint2*>(dst) = r;
    if (MODE == 2) {
      uint2 l;
      l.x = bn_pack_bf16x2(a0 - bn_bf16_round(a0), a1 - bn_bf16_round(a1));
      l.y = bn_pack_bf16x2(a2 - bn_bf16_round(a2), a3 - bn_bf16_round(a3));
      *reinterpret_cast<uint2*>(dst + C) = l;
    }
  };
  // U elements per thread and iteration, loads first
  for (; i + (U - 1) * nthreads < n4; i += U * nthreads, pix += U * pix_step) {
    float4 g[U], v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) g[u] = __ldcs(gz + i + u * nthreads);
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = load_y4<I16>(y, i + u * nthreads);
#pragma unroll
    for (int u = 0; u < U; ++u) emit(pix + u * pix_step, g[u], v[u]);
  }
  for (; i < n4; i += nthreads, pix += pix_step) emit(pix, __ldcs(gz + i), load_y4<I16>(y, i));
}

static int bn_grid(int64_t work, int C4, int per_sm = 8) {
  // grid whose thread count is a multiple of C4 (C4 in {4,..,128} divides 256*k); per_sm blocks per SM at most
  int64_t blocks = (work + kBnThreads - 1) / kBnThreads;
  const int64_t cap = int64_t(num_sms()) * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  while ((blocks * kBnThreads) % C4 != 0) ++blocks;
  return int(blocks);
}

// Forward statistics pass (also the fallback of conv kernels without a statistics epilogue).
int bn_stats_launch(const float* y, int64_t n_pix, int C, double* sums, uint32_t* ymax, cudaStream_t st) {
  BDBNN_REQUIRE(C > 0 && (C & 3) == 0 && C <= 4096, "bn_stats: C must be a multiple of 4, <= 4096");
  const int C4 = C / 4;
  BDBNN_CUDA(bn_reduce_allow(bn_reduce_kernel<false>, C));
  bn_reduce_kernel<false><<<bn_grid(n_pix * C4 / 8, C4, n_pix * C4 > (int64_t(16) << 20) ? 8 : 3), kBnThreads,
                            bn_reduce_smem(C), st>>>(reinterpret_cast<const float4*>(y), nullptr, nullptr,
                                                                 nullptr, n_pix, C4, sums, ymax);
  return check_launch("bn_reduce_kernel<fwd>");
}

}  // namespace bdbnn

using namespace bdbnn;

static int bn_dims_ok(int64_t n_pix, int32_t C, bool pack) {
  BDBNN_REQUIRE(n_pix > 0 && C > 0 && (C & 3) == 0, "bn: C must be a positive multiple of 4");
  BDBNN_REQUIRE(C <= 4096, "bn: C too large");
  BDBNN_REQUIRE(!pack || (C & 31) == 0, "bn: packing needs C %% 32 == 0");
  return BDBNN_OK;
}

static int bn_fwd_impl(const void* y, const float* alpha_i16, const float* residual, const float* gamma,
                       const float* beta, int64_t n_pix, int32_t C, float eps, float momentum, float* running_mean,
                       float* running_var, double* sums_ws, uint32_t* ymax_bits, float* mean, float* invstd,
                       float* ab_ws, float* z, uint32_t* sign_bits, uint32_t* mask_bits, uint16_t* xb,
                       uint8_t* xb_fp8, int32_t fmt, int32_t stats_ready, void* stream) {
  const bool pack = sign_bits != nullptr;
  const bool i16 = alpha_i16 != nullptr;
  BDBNN_REQUIRE(!i16 || stats_ready, "bn_fwd_i16: the statistics must come from the conv epilogue (stats_ready = 1)");
  int rc = bn_dims_ok(n_pix, C, pack);
  if (rc) return rc;
  BDBNN_REQUIRE(y && gamma && beta && sums_ws && ymax_bits && mean && invstd && ab_ws && z, "bn_fwd: NULL pointer");
  BDBNN_REQUIRE(!pack || (mask_bits && xb), "bn_fwd: packing needs sign_bits, mask_bits and xb");
  BDBNN_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "bn_fwd: running stats come in pairs");
  cudaStream_t st = cudaStream_t(stream);
  const int C4 = C / 4;
  if (!stats_ready) {          // else: sums_ws / ymax_bits were filled by the conv's epilogue
    BDBNN_CUDA(cudaMemsetAsync(sums_ws, 0, size_t(2 * C) * sizeof(double), st));
    BDBNN_CUDA(cudaMemsetAsync(ymax_bits, 0, size_t(C) * sizeof(uint32_t), st));
    rc = bn_stats_launch(static_cast<const float*>(y), n_pix, C, sums_ws, ymax_bits, st);
    if (rc) return rc;
  }
  float* a = ab_ws;
  float* b = ab_ws + C;
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums_ws, n_pix, C, eps, gamma, beta, mean, invstd, a, b,
                                                       running_mean, running_var, momentum, alpha_i16);
  rc = check_launch("bn_finalize_kernel");
  if (rc) return rc;
  const int64_t n4 = n_pix * C4;
  const int grid = bn_grid(n4, C4);
  const float4* r4 = reinterpret_cast<const float4*>(residual);
  float4* z4 = reinterpret_cast<float4*>(z);
  if (pack) {
    const uint32_t one16 = fmt == BDBNN_FMT_FP16 ? 0x3C00u : 0x3F80u;
    uint2* xb2 = reinterpret_cast<uint2*>(xb);
    uint32_t* xb8 = reinterpret_cast<uint32_t*>(xb_fp8);
    // four float4 per thread and iteration (measured: bn_fwd 1.13 -> 1.04 ms per ResNet-18 step vs two); BDBNN_BN_UNROLL=2
    static const int unroll2 = [] { const char* e = getenv("BDBNN_BN_UNROLL"); return e ? atoi(e) == 2 : 0; }();
    if (i16 && unroll2)
      bn_apply_add_pack_kernel<true, true, 2><<<grid, kBnThreads, 0, st>>>(y, r4, a, b, n4, C4, z4, sign_bits, mask_bits,
                                                                            xb2, xb8, one16);
    else if (i16)
      bn_apply_add_pack_kernel<true, true><<<grid, kBnThreads, 0, st>>>(y, r4, a, b, n4, C4, z4, sign_bits, mask_bits,
                                                                         xb2, xb8, one16);
    else
      bn_apply_add_pack_kernel<true, false><<<grid, kBnThreads, 0, st>>>(y, r4, a, b, n4, C4, z4, sign_bits, mask_bits,
                                                                          xb2, xb8, one16);
  } else {
    if (i16)
      bn_apply_add_pack_kernel<false, true><<<grid, kBnThreads, 0, st>>>(y, r4, a, b, n4, C4, z4, nullptr, nullptr,
                                                                          nullptr, nullptr, 0u);
    else
      bn_apply_add_pack_kernel<false, false><<<grid, kBnThreads, 0, st>>>(y, r4, a, b, n4, C4, z4, nullptr, nullptr,
                                                                           nullptr, nullptr, 0u);
  }
  return check_launch("bn_apply_add_pack_kernel");
}

extern "C" int bdbnn_bn_fwd(const float* y, const float* residual, const float* gamma, const float* beta,
                            int64_t n_pix, int32_t C, float eps, float momentum, float* running_mean,
                            float* running_var, double* sums_ws, uint32_t* ymax_bits, float* mean,
                            float* invstd, float* ab_ws, float* z, uint32_t* sign_bits, uint32_t* mask_bits,
                            uint16_t* xb, uint8_t* xb_fp8, int32_t fmt, int32_t stats_ready, void* stream) {
  return bn_fwd_impl(y, nullptr, residual, gamma, beta, n_pix, C, eps, momentum, running_mean, running_var, sums_ws,
                     ymax_bits, mean, invstd, ab_ws, z, sign_bits, mask_bits, xb, xb_fp8, fmt, stats_ready, stream);
}

extern "C" int bdbnn_bn_fwd_i16(const int16_t* y_int, const float* alpha, const float* residual, const float* gamma,
                                const float* beta, int64_t n_pix, int32_t C, float eps, float momentum,
                                float* running_mean, float* running_var, double* sums_ws, uint32_t* ymax_bits,
                                float* mean, float* invstd, float* ab_ws, float* z, uint32_t* sign_bits,
                                uint32_t* mask_bits, uint16_t* xb, uint8_t* xb_fp8, int32_t fmt, void* stream) {
  BDBNN_REQUIRE(alpha != nullptr, "bn_fwd_i16: NULL alpha");
  return bn_fwd_impl(y_int, alpha, residual, gamma, beta, n_pix, C, eps, momentum, running_mean, running_var, sums_ws,
                     ymax_bits, mean, invstd, ab_ws, z, sign_bits, mask_bits, xb, xb_fp8, fmt, 1, stream);
}

static int bn_bwd_pack_impl(const float* gz, const void* y, const float* alpha_i16, const float* mean,
                            const float* invstd, const float* gamma, const float* gscale, const uint32_t* ymax_bits,
                            int64_t n_pix, int32_t C, int32_t grad_mode, double* sums_ws, uint32_t* gmax_bits,
                            float* consts_ws, float* dgamma, float* dbeta, uint32_t* amax_bits, uint16_t* gys,
                            int stats_ready, void* stream) {
  const bool i16 = alpha_i16 != nullptr;
  int rc = bn_dims_ok(n_pix, C, false);
  if (rc) return rc;
  BDBNN_REQUIRE(gz && y && mean && invstd && gamma && gscale && ymax_bits && sums_ws && gmax_bits && consts_ws &&
                    dgamma && dbeta && amax_bits && gys,
                "bn_bwd_pack: NULL pointer");
  BDBNN_REQUIRE(grad_mode >= BDBNN_GRAD_BF16 && grad_mode <= BDBNN_GRAD_FP16S, "bn_bwd_pack: bad grad_mode");
  cudaStream_t st = cudaStream_t(stream);
  const int C4 = C / 4;
  if (!stats_ready) {       // else: sums_ws / gmax_bits were filled by the dgrad epilogue that produced gz
    BDBNN_CUDA(cudaMemsetAsync(sums_ws, 0, size_t(2 * C) * sizeof(double), st));
    BDBNN_CUDA(cudaMemsetAsync(gmax_bits, 0, size_t(C) * sizeof(uint32_t), st));
    const int rgrid = bn_grid(n_pix * C4 / 8, C4, n_pix * C4 > (int64_t(16) << 20) ? 8 : 3);
    BDBNN_CUDA(i16 ? bn_reduce_allow(bn_reduce_kernel<true, true>, C) : bn_reduce_allow(bn_reduce_kernel<true, false>, C));
    if (i16)
      bn_reduce_kernel<true, true><<<rgrid, kBnThreads, bn_reduce_smem(C), st>>>(
          reinterpret_cast<const float4*>(gz), y, mean, invstd, n_pix, C4, sums_ws, gmax_bits, alpha_i16);
    else
      bn_reduce_kernel<true, false><<<rgrid, kBnThreads, bn_reduce_smem(C), st>>>(
          reinterpret_cast<const float4*>(gz), y, mean, invstd, n_pix, C4, sums_ws, gmax_bits, nullptr);
    rc = check_launch("bn_reduce_kernel<bwd>");
    if (rc) return rc;
  }
  bn_bwd_bound_kernel<<<1, 256, 0, st>>>(sums_ws, gmax_bits, ymax_bits, n_pix, C, mean, invstd, gamma, gscale,
                                         reinterpret_cast<float4*>(consts_ws), dgamma, dbeta, amax_bits, 1.0f,
                                         alpha_i16);
  rc = check_launch("bn_bwd_bound_kernel");
  if (rc) return rc;
  const int64_t n4 = n_pix * C4;
  // BDBNN_BN_BWD_PER_SM: resident blocks per SM of the backward apply kernel (64 registers x 256 threads: 4 fill the
  // register file; 3 leave room for a side-stream wgrad CTA next to them)
  static const int bwd_per_sm = [] { const char* e = getenv("BDBNN_BN_BWD_PER_SM"); return e ? atoi(e) : 8; }();
  const int grid = bn_grid(n4, C4, bwd_per_sm);
  const float4* g4 = reinterpret_cast<const float4*>(gz);
  const float4* k4 = reinterpret_cast<const float4*>(consts_ws);
  if (i16) {
    if (grad_mode == BDBNN_GRAD_FP16S)
      bn_bwd_pack_kernel<3, true><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
    else if (grad_mode == BDBNN_GRAD_BF16X2)
      bn_bwd_pack_kernel<2, true><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
    else
      bn_bwd_pack_kernel<1, true><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
  } else {
    if (grad_mode == BDBNN_GRAD_FP16S)
      bn_bwd_pack_kernel<3, false><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
    else if (grad_mode == BDBNN_GRAD_BF16X2)
      bn_bwd_pack_kernel<2, false><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
    else
      bn_bwd_pack_kernel<1, false><<<grid, kBnThreads, 0, st>>>(g4, y, k4, amax_bits, n4, C4, gys);
  }
  return check_launch("bn_bwd_pack_kernel");
}

extern "C" int bdbnn_bn_bwd_pack(const float* gz, const float* y, const float* mean, const float* invstd,
                                 const float* gamma, const float* gscale, const uint32_t* ymax_bits,
                                 int64_t n_pix, int32_t C, int32_t grad_mode, double* sums_ws,
                                 uint32_t* gmax_bits, float* consts_ws, float* dgamma, float* dbeta,
                                 uint32_t* amax_bits, uint16_t* gys, void* stream) {
  return bn_bwd_pack_impl(gz, y, nullptr, mean, invstd, gamma, gscale, ymax_bits, n_pix, C, grad_mode, sums_ws,
                          gmax_bits, consts_ws, dgamma, dbeta, amax_bits, gys, 0, stream);
}

extern "C" int bdbnn_bn_bwd_pack_i16(const float* gz, const int16_t* y_int, const float* alpha, const float* mean,
                                     const float* invstd, const float* gamma, const float* gscale,
                                     const uint32_t* ymax_bits, int64_t n_pix, int32_t C, int32_t grad_mode,
                                     double* sums_ws, uint32_t* gmax_bits, float* consts_ws, float* dgamma,
                                     float* dbeta, uint32_t* amax_bits, uint16_t* gys, int32_t stats_ready,
                                     void* stream) {
  BDBNN_REQUIRE(alpha != nullptr, "bn_bwd_pack_i16: NULL alpha");
  return bn_bwd_pack_impl(gz, y_int, alpha, mean, invstd, gamma, gscale, ymax_bits, n_pix, C, grad_mode, sums_ws,
                          gmax_bits, consts_ws, dgamma, dbeta, amax_bits, gys, stats_ready, stream);
}

// ===================================================================================================
// Stem: BatchNorm(train) + MaxPool fused (the 112x112x64 stem activation is the largest tensor of the
// step: 822 MB at N=256).  The BN output is never materialised:
//   forward : bn_reduce<fwd>(y) -> bn_finalize -> bn_pool_fwd: z = maxpool(a*y+b) + winner index +
//             y at the winner (for the backward's yhat) [+ the first binary conv's sign/mask/+-1 packs]
//   backward: bn_reduce<bwd>(g_pool, y_sel) over the POOLED tensors (every pooled gradient lands on
//             exactly one input position, so sum gz = sum g_pool and sum gz*yhat = sum g_pool*yhat_sel)
//             -> bn_bwd_bound -> bn_pool_bwd: gy = a*(gz - m1 - yhat*m2) for every input position, with
//             gz gathered from the (<= 4) windows whose winner is that position.
// torch.nn.MaxPool2d semantics on the BN output (first maximum in scan order wins, NaN propagates).
// ===================================================================================================
namespace bdbnn {

template <bool PACK>
__global__ void __launch_bounds__(kBnThreads)
bn_pool_fwd_kernel(const float4* __restrict__ y, const float* __restrict__ a, const float* __restrict__ b,
                   int N, int H, int W, int C4, int Ho, int Wo, int k, int s, int p, int64_t total,
                   float4* __restrict__ z, float4* __restrict__ ysel, uint32_t* __restrict__ idx,
                   uint32_t* __restrict__ sign_bits, uint32_t* __restrict__ mask_bits, uint2* __restrict__ xb4,
                   uint32_t* __restrict__ xb8, uint32_t one16) {
  const int lane = threadIdx.x & 31;
  const uint32_t group_mask = 0xffu << (lane & 24);
  const int sh = (lane & 7) * 4;
  const uint32_t pos = one16, neg = one16 | 0x8000u;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;     // multiple of C4
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c = int(i % C4);
  const float4 av = *reinterpret_cast<const float4*>(a + c * 4);
  const float4 bv = *reinterpret_cast<const float4*>(b + c * 4);
  for (; i < total; i += nthreads) {
    int64_t q = i / C4;
    const int wo = int(q % Wo); q /= Wo;
    const int ho = int(q % Ho);
    const int n = int(q / Ho);
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f), ys = m;
    uint32_t w4 = 0;
    bool first = true;
    for (int r = 0; r < k; ++r) {
      const int h = ho * s - p + r;
      if (h < 0 || h >= H) continue;
      for (int t = 0; t < k; ++t) {
        const int w = wo * s - p + t;
        if (w < 0 || w >= W) continue;
        const float4 yv = __ldg(y + ((int64_t(n) * H + h) * W + w) * C4 + c);
        const float4 v = make_float4(fmaf(yv.x, av.x, bv.x), fmaf(yv.y, av.y, bv.y), fmaf(yv.z, av.z, bv.z),
                                     fmaf(yv.w, av.w, bv.w));
        const uint32_t tap = uint32_t(r * k + t);
        if (first || v.x > m.x || v.x != v.x) { m.x = v.x; ys.x = yv.x; w4 = (w4 & 0xffffff00u) | tap; }
        if (first || v.y > m.y || v.y != v.y) { m.y = v.y; ys.y = yv.y; w4 = (w4 & 0xffff00ffu) | (tap << 8); }
        if (first || v.z > m.z || v.z != v.z) { m.z = v.z; ys.z = yv.z; w4 = (w4 & 0xff00ffffu) | (tap << 16); }
        if (first || v.w > m.w || v.w != v.w) { m.w = v.w; ys.w = yv.w; w4 = (w4 & 0x00ffffffu) | (tap << 24); }
        first = false;
      }
    }
    z[i] = m;
    ysel[i] = ys;
    idx[i] = w4;
    if (PACK) {
      const uint32_t s0 = m.x >= 0.0f, s1 = m.y >= 0.0f, s2 = m.z >= 0.0f, s3 = m.w >= 0.0f;
      const uint32_t m0 = fabsf(m.x) <= 1.0f, m1 = fabsf(m.y) <= 1.0f, m2 = fabsf(m.z) <= 1.0f,
                     m3 = fabsf(m.w) <= 1.0f;
      const uint32_t sw = __reduce_or_sync(group_mask, (s0 | (s1 << 1) | (s2 << 2) | (s3 << 3)) << sh);
      const uint32_t mw = __reduce_or_sync(group_mask, (m0 | (m1 << 1) | (m2 << 2) | (m3 << 3)) << sh);
      if ((lane & 7) == 0) {
        sign_bits[i >> 3] = sw;
        mask_bits[i >> 3] = mw;
      }
      uint2 o;
      o.x = (s0 ? pos : neg) | ((s1 ? pos : neg) << 16);
      o.y = (s2 ? pos : neg) | ((s3 ? pos : neg) << 16);
      xb4[i] = o;
      if (xb8 != nullptr)
        xb8[i] = 0x38383838u | ((s0 ? 0u : 0x80u) | (s1 ? 0u : 0x8000u) | (s2 ? 0u : 0x800000u) | (s3 ? 0u : 0x80000000u));
    }
  }
}

// 3x3 / stride-2 / pad-1 forward (the stem's pool) with one block per output row (n, ho): the three input
// row pointers and the row validity are per block, the tap loop is unrolled, and the winner index is kept
// as four small integers instead of read-modify-write byte lanes — about half the instructions of the
// generic kernel, which ncu showed issue-bound (55-60 % issue-slot utilisation at 2.4 TB/s).
// Same scan order and NaN rule, so outputs are bit-identical.  blockDim.x is a multiple of C4.
template <bool PACK>
__global__ void __launch_bounds__(kBnThreads)
bn_pool_fwd_k3s2_kernel(const float4* __restrict__ y, const float* __restrict__ a, const float* __restrict__ b,
                        int H, int W, int C4, int Ho, int Wo, float4* __restrict__ z, float4* __restrict__ ysel,
                        uint32_t* __restrict__ idx, uint32_t* __restrict__ sign_bits,
                        uint32_t* __restrict__ mask_bits, uint2* __restrict__ xb4, uint32_t* __restrict__ xb8,
                        uint32_t one16) {
  const int lane = threadIdx.x & 31;
  const uint32_t group_mask = 0xffu << (lane & 24);
  const int sh = (lane & 7) * 4;
  const uint32_t pos = one16, neg = one16 | 0x8000u;
  const int c = threadIdx.x % C4;
  const float4 av = *reinterpret_cast<const float4*>(a + c * 4);
  const float4 bv = *reinterpret_cast<const float4*>(b + c * 4);
  const int n = blockIdx.x / Ho, ho = blockIdx.x - n * Ho;
  const int h0 = 2 * ho - 1;
  const float4* rows[3];
  bool rok[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int h = h0 + r;
    rok[r] = h >= 0 && h < H;
    rows[r] = y + (int64_t(n) * H + (rok[r] ? h : 0)) * W * C4 + c;
  }
  const int per_row = Wo * C4;               // multiple of 8 when PACK (C % 32 == 0)
  const int64_t out0 = (int64_t(n) * Ho + ho) * per_row;
  for (int j = threadIdx.x; j < per_row; j += blockDim.x) {
    const int wo = j / C4;
    const int w0 = 2 * wo - 1;
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f), ys = m;
    uint32_t tx = 0, ty = 0, tz = 0, tw = 0;
    bool first = true;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      if (!rok[r]) continue;
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const int w = w0 + t;
        if (w < 0 || w >= W) continue;
        const float4 yv = __ldg(rows[r] + int64_t(w) * C4);
        const float4 v = make_float4(fmaf(yv.x, av.x, bv.x), fmaf(yv.y, av.y, bv.y), fmaf(yv.z, av.z, bv.z),
                                     fmaf(yv.w, av.w, bv.w));
        const uint32_t tap = uint32_t(r * 3 + t);
        if (first || v.x > m.x || v.x != v.x) { m.x = v.x; ys.x = yv.x; tx = tap; }
        if (first || v.y > m.y || v.y != v.y) { m.y = v.y; ys.y = yv.y; ty = tap; }
        if (first || v.z > m.z || v.z != v.z) { m.z = v.z; ys.z = yv.z; tz = tap; }
        if (first || v.w > m.w || v.w != v.w) { m.w = v.w; ys.w = yv.w; tw = tap; }
        first = false;
      }
    }
    const int64_t i = out0 + j;
    z[i] = m;
    ysel[i] = ys;
    idx[i] = tx | (ty << 8) | (tz << 16) | (tw << 24);
    if (PACK) {
      const uint32_t s0 = m.x >= 0.0f, s1 = m.y >= 0.0f, s2 = m.z >= 0.0f, s3 = m.w >= 0.0f;
      const uint32_t m0 = fabsf(m.x) <= 1.0f, m1 = fabsf(m.y) <= 1.0f, m2 = fabsf(m.z) <= 1.0f,
                     m3 = fabsf(m.w) <= 1.0f;
      const uint32_t sw = __reduce_or_sync(group_mask, (s0 | (s1 << 1) | (s2 << 2) | (s3 << 3)) << sh);
      const uint32_t mw = __reduce_or_sync(group_mask, (m0 | (m1 << 1) | (m2 << 2) | (m3 << 3)) << sh);
      if ((lane & 7) == 0) {
        sign_bits[i >> 3] = sw;
        mask_bits[i >> 3] = mw;
      }
      uint2 o;
      o.x = (s0 ? pos : neg) | ((s1 ? pos : neg) << 16);
      o.y = (s2 ? pos : neg) | ((s3 ? pos : neg) << 16);
      xb4[i] = o;
      if (xb8 != nullptr)
        xb8[i] = 0x38383838u | ((s0 ? 0u : 0x80u) | (s1 ? 0u : 0x8000u) | (s2 ? 0u : 0x800000u) | (s3 ? 0u : 0x80000000u));
    }
  }
}

// gy[n,h,w,c] = A*(gz - m1 - (y-mean)*m2'),  gz = sum of g_pool over the windows won by (h,w);
// consts[c] = {m1, m2*invstd, mean, A} from bn_bwd_bound_kernel (gscale = 1).
// HALF: write gys = fp16(gy * 2^e) (e from the bound in amax_bits: the stem conv's wgrad operand, so the
// 4-byte gradient of the largest activation of the step is never written) instead of fp32 gy.
template <bool HALF>
__global__ void __launch_bounds__(kBnThreads)
bn_pool_bwd_kernel(const float4* __restrict__ gpool, const uint32_t* __restrict__ idx, const float4* __restrict__ y,
                   const float4* __restrict__ consts, int N, int H, int W, int C4, int Ho, int Wo, int k, int s,
                   int p, int64_t total, float4* __restrict__ gy, const uint32_t* __restrict__ amax_bits,
                   uint2* __restrict__ gys) {
  const float up = HALF ? amax_pow2_scale(__ldg(amax_bits), false) : 1.0f;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;     // multiple of C4
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c = int(i % C4);
  const float4 k0 = consts[c * 4 + 0], k1 = consts[c * 4 + 1], k2 = consts[c * 4 + 2], k3 = consts[c * 4 + 3];
  for (; i < total; i += nthreads) {
    int64_t q = i / C4;
    const int w = int(q % W); q /= W;
    const int h = int(q % H);
    const int n = int(q / H);
    float4 gz = make_float4(0.f, 0.f, 0.f, 0.f);
    int ho0 = (h + p - k + s) / s;
    if (h + p - k + 1 <= 0) ho0 = 0;
    int wo0 = (w + p - k + s) / s;
    if (w + p - k + 1 <= 0) wo0 = 0;
    const int ho1 = min((h + p) / s, Ho - 1), wo1 = min((w + p) / s, Wo - 1);
    for (int ho = ho0; ho <= ho1; ++ho) {
      const uint32_t r = uint32_t(h - (ho * s - p));
      for (int wo = wo0; wo <= wo1; ++wo) {
        const uint32_t tap = r * uint32_t(k) + uint32_t(w - (wo * s - p));
        const int64_t o = ((int64_t(n) * Ho + ho) * Wo + wo) * C4 + c;
        const uint32_t w4 = __ldg(idx + o);
        const float4 g = __ldg(gpool + o);
        if ((w4 & 0xffu) == tap) gz.x += g.x;
        if (((w4 >> 8) & 0xffu) == tap) gz.y += g.y;
        if (((w4 >> 16) & 0xffu) == tap) gz.z += g.z;
        if ((w4 >> 24) == tap) gz.w += g.w;
      }
    }
    const float4 v = __ldcs(y + i);
    float4 o;
    o.x = (gz.x - k0.x - (v.x - k0.z) * k0.y) * k0.w;
    o.y = (gz.y - k1.x - (v.y - k1.z) * k1.y) * k1.w;
    o.z = (gz.z - k2.x - (v.z - k2.z) * k2.y) * k2.w;
    o.w = (gz.w - k3.x - (v.w - k3.z) * k3.y) * k3.w;
    if (HALF) {
      const __half2 h0 = __floats2half2_rn(o.x * up, o.y * up), h1 = __floats2half2_rn(o.z * up, o.w * up);
      gys[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
    } else {
      gy[i] = o;
    }
  }
}

// Same result for the 3x3 / stride-2 / pad-1 pool (the stem's), restructured so that one thread owns a 2x2
// block of input positions (rows 2a, 2a+1; columns 2b, 2b+1) of one channel quad: the four positions are
// covered by the same four pooling windows (a..a+1, b..b+1), so each window's winner word and gradient
// are loaded once for four outputs (the generic kernel re-reads them 2.25x per output on average) and
// the index arithmetic is per block, not per element.  Windows are visited in the generic kernel's
// order, so the sums are bit-identical.  blockDim.x must be a multiple of C4.
template <bool HALF>
__global__ void __launch_bounds__(kBnThreads)
bn_pool_bwd_k3s2_kernel(const float4* __restrict__ gpool, const uint32_t* __restrict__ idx,
                        const float4* __restrict__ y, const float4* __restrict__ consts, int H, int W, int C4,
                        int Ho, int Wo, int HB, int WB, float4* __restrict__ gy,
                        const uint32_t* __restrict__ amax_bits, uint2* __restrict__ gys) {
  const float up = HALF ? amax_pow2_scale(__ldg(amax_bits), false) : 1.0f;
  const int c = threadIdx.x % C4;
  const float4 k0 = consts[c * 4 + 0], k1 = consts[c * 4 + 1], k2 = consts[c * 4 + 2], k3 = consts[c * 4 + 3];
  const int n = blockIdx.x / HB, a = blockIdx.x - n * HB;
  const int h0 = 2 * a, h1 = 2 * a + 1;
  const int per_row = WB * C4;
  for (int j = threadIdx.x; j < per_row; j += blockDim.x) {
    const int b = j / C4;
    const int w0 = 2 * b, w1 = 2 * b + 1;
    // windows (a,b) (a,b+1) (a+1,b) (a+1,b+1)
    float4 g[4];
    uint32_t wd[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int ho = a + (q >> 1), wo = b + (q & 1);
      if (ho < Ho && wo < Wo) {
        const int64_t o = ((int64_t(n) * Ho + ho) * Wo + wo) * C4 + c;
        wd[q] = __ldg(idx + o);
        g[q] = __ldg(gpool + o);
      } else {
        wd[q] = 0xffffffffu;                      // tap 255 never matches
        g[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    auto pick = [&](float4& acc, int q, uint32_t tap) {
      const uint32_t w4 = wd[q];
      if ((w4 & 0xffu) == tap) acc.x += g[q].x;
      if (((w4 >> 8) & 0xffu) == tap) acc.y += g[q].y;
      if (((w4 >> 16) & 0xffu) == tap) acc.z += g[q].z;
      if ((w4 >> 24) == tap) acc.w += g[q].w;
    };
    float4 z00 = make_float4(0.f, 0.f, 0.f, 0.f), z01 = z00, z10 = z00, z11 = z00;
    pick(z00, 0, 4u);                                             // (2a  , 2b  ): centre of window (a,b)
    pick(z01, 0, 5u); pick(z01, 1, 3u);                           // (2a  , 2b+1)
    pick(z10, 0, 7u); pick(z10, 2, 1u);                           // (2a+1, 2b  )
    pick(z11, 0, 8u); pick(z11, 1, 6u); pick(z11, 2, 2u); pick(z11, 3, 0u);
    auto emit = [&](int h, int w, const float4& gz) {
      if (h >= H || w >= W) return;
      const int64_t i = ((int64_t(n) * H + h) * W + w) * C4 + c;
      const float4 v = __ldcs(y + i);
      float4 o;
      o.x = (gz.x - k0.x - (v.x - k0.z) * k0.y) * k0.w;
      o.y = (gz.y - k1.x - (v.y - k1.z) * k1.y) * k1.w;
      o.z = (gz.z - k2.x - (v.z - k2.z) * k2.y) * k2.w;
      o.w = (gz.w - k3.x - (v.w - k3.z) * k3.y) * k3.w;
      if (HALF) {
        const __half2 p0 = __floats2half2_rn(o.x * up, o.y * up), p1 = __floats2half2_rn(o.z * up, o.w * up);
        gys[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&p0), *reinterpret_cast<const uint32_t*>(&p1));
      } else {
        gy[i] = o;
      }
    };
    emit(h0, w0, z00);
    emit(h0, w1, z01);
    emit(h1, w0, z10);
    emit(h1, w1, z11);
  }
}

}  // namespace bdbnn

using namespace bdbnn;

static int pool_geom_ok(int N, int H, int W, int C, int k, int s, int p, int Ho, int Wo) {
  BDBNN_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && (C & 3) == 0 && C <= 4096, "bn_pool: bad N/H/W/C");
  BDBNN_REQUIRE(k > 0 && k <= 15 && s > 0 && p >= 0 && 2 * p <= k, "bn_pool: bad k/stride/pad");
  BDBNN_REQUIRE(Ho == (H + 2 * p - k) / s + 1 && Wo == (W + 2 * p - k) / s + 1 && Ho > 0 && Wo > 0,
                "bn_pool: inconsistent output size");
  return BDBNN_OK;
}

extern "C" int bdbnn_bn_pool_fwd(const float* y, const float* gamma, const float* beta, int32_t N, int32_t H,
                                 int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad, int32_t Ho,
                                 int32_t Wo, float eps, float momentum, float* running_mean, float* running_var,
                                 double* sums_ws, uint32_t* ymax_bits, float* mean, float* invstd, float* ab_ws,
                                 float* z, float* y_sel, uint8_t* idx, uint32_t* sign_bits, uint32_t* mask_bits,
                                 uint16_t* xb, uint8_t* xb_fp8, int32_t fmt, int32_t stats_ready, void* stream) {
  int rc = pool_geom_ok(N, H, W, C, k, stride, pad, Ho, Wo);
  if (rc) return rc;
  const bool pack = sign_bits != nullptr;
  BDBNN_REQUIRE(y && gamma && beta && sums_ws && ymax_bits && mean && invstd && ab_ws && z && y_sel && idx,
                "bn_pool_fwd: NULL pointer");
  BDBNN_REQUIRE(!pack || ((C & 31) == 0 && mask_bits && xb), "bn_pool_fwd: packing needs C %% 32 == 0 and all pack outputs");
  cudaStream_t st = cudaStream_t(stream);
  const int C4 = C / 4;
  const int64_t n_pix = int64_t(N) * H * W;
  if (!stats_ready) {
    BDBNN_CUDA(cudaMemsetAsync(sums_ws, 0, size_t(2 * C) * sizeof(double), st));
    BDBNN_CUDA(cudaMemsetAsync(ymax_bits, 0, size_t(C) * sizeof(uint32_t), st));
    rc = bn_stats_launch(y, n_pix, C, sums_ws, ymax_bits, st);
    if (rc) return rc;
  }
  float* a = ab_ws;
  float* b = ab_ws + C;
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums_ws, n_pix, C, eps, gamma, beta, mean, invstd, a, b,
                                                       running_mean, running_var, momentum);
  rc = check_launch("bn_finalize_kernel");
  if (rc) return rc;
  const int64_t total = int64_t(N) * Ho * Wo * C4;
  const int grid = bn_grid(total, C4);
  const float4* y4 = reinterpret_cast<const float4*>(y);
  // PACK needs the 8 lanes of a 32-channel word inside one iteration of one warp: per-row work and the
  // block size must be multiples of 8 quads, which C % 32 == 0 gives when blockDim is a multiple of C4
  if (k == 3 && stride == 2 && pad == 1 && C4 <= kBnThreads && (!pack || (C4 % 8 == 0 && kBnThreads % C4 == 0))) {
    const int threads = (kBnThreads / C4) * C4;
    const unsigned rows_grid = unsigned(N) * unsigned(Ho);
    if (pack)
      bn_pool_fwd_k3s2_kernel<true><<<rows_grid, threads, 0, st>>>(
          y4, a, b, H, W, C4, Ho, Wo, reinterpret_cast<float4*>(z), reinterpret_cast<float4*>(y_sel),
          reinterpret_cast<uint32_t*>(idx), sign_bits, mask_bits, reinterpret_cast<uint2*>(xb),
          reinterpret_cast<uint32_t*>(xb_fp8), fmt == BDBNN_FMT_FP16 ? 0x3C00u : 0x3F80u);
    else
      bn_pool_fwd_k3s2_kernel<false><<<rows_grid, threads, 0, st>>>(
          y4, a, b, H, W, C4, Ho, Wo, reinterpret_cast<float4*>(z), reinterpret_cast<float4*>(y_sel),
          reinterpret_cast<uint32_t*>(idx), nullptr, nullptr, nullptr, nullptr, 0u);
    return check_launch("bn_pool_fwd_k3s2_kernel");
  }
  if (pack) {
    bn_pool_fwd_kernel<true><<<grid, kBnThreads, 0, st>>>(
        y4, a, b, N, H, W, C4, Ho, Wo, k, stride, pad, total, reinterpret_cast<float4*>(z),
        reinterpret_cast<float4*>(y_sel), reinterpret_cast<uint32_t*>(idx), sign_bits, mask_bits,
        reinterpret_cast<uint2*>(xb), reinterpret_cast<uint32_t*>(xb_fp8), fmt == BDBNN_FMT_FP16 ? 0x3C00u : 0x3F80u);
  } else {
    bn_pool_fwd_kernel<false><<<grid, kBnThreads, 0, st>>>(
        y4, a, b, N, H, W, C4, Ho, Wo, k, stride, pad, total, reinterpret_cast<float4*>(z),
        reinterpret_cast<float4*>(y_sel), reinterpret_cast<uint32_t*>(idx), nullptr, nullptr, nullptr, nullptr, 0u);
  }
  return check_launch("bn_pool_fwd_kernel");
}

extern "C" int bdbnn_bn_pool_bwd(const float* g_pool, const uint8_t* idx, const float* y, const float* y_sel,
                                 const float* mean, const float* invstd, const float* gamma, const float* ones,
                                 const uint32_t* ymax_bits, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k,
                                 int32_t stride, int32_t pad, int32_t Ho, int32_t Wo, double* sums_ws,
                                 uint32_t* gmax_bits, float* consts_ws, float* dgamma, float* dbeta,
                                 uint32_t* amax_scratch, float* gy, uint16_t* gys, void* stream) {
  int rc = pool_geom_ok(N, H, W, C, k, stride, pad, Ho, Wo);
  if (rc) return rc;
  BDBNN_REQUIRE(g_pool && idx && y && y_sel && mean && invstd && gamma && ones && ymax_bits && sums_ws && gmax_bits &&
                    consts_ws && dgamma && dbeta && amax_scratch && (gy || gys),
                "bn_pool_bwd: NULL pointer");
  cudaStream_t st = cudaStream_t(stream);
  const int C4 = C / 4;
  const int64_t n_pool = int64_t(N) * Ho * Wo, n_full = int64_t(N) * H * W;
  BDBNN_CUDA(cudaMemsetAsync(sums_ws, 0, size_t(2 * C) * sizeof(double), st));
  BDBNN_CUDA(cudaMemsetAsync(gmax_bits, 0, size_t(C) * sizeof(uint32_t), st));
  BDBNN_CUDA(bn_reduce_allow(bn_reduce_kernel<true>, C));
  bn_reduce_kernel<true><<<bn_grid(n_pool * C4 / 8, C4, 3), kBnThreads, bn_reduce_smem(C), st>>>(
      reinterpret_cast<const float4*>(g_pool), reinterpret_cast<const float4*>(y_sel), mean, invstd, n_pool, C4,
      sums_ws, gmax_bits);
  rc = check_launch("bn_reduce_kernel<bwd,pool>");
  if (rc) return rc;
  // means are over the FULL-resolution element count; gscale = 1 (`ones`)
  const int per_dim = (k + stride - 1) / stride;          // pooling windows covering one position, per axis
  bn_bwd_bound_kernel<<<1, 256, 0, st>>>(sums_ws, gmax_bits, ymax_bits, n_full, C, mean, invstd, gamma, ones,
                                         reinterpret_cast<float4*>(consts_ws), dgamma, dbeta, amax_scratch,
                                         float(per_dim * per_dim));
  rc = check_launch("bn_bwd_bound_kernel");
  if (rc) return rc;
  const int64_t total = n_full * C4;
  if (k == 3 && stride == 2 && pad == 1 && C4 <= kBnThreads) {
    const int HB = (H + 1) / 2, WB = (W + 1) / 2;
    const int threads = (kBnThreads / C4) * C4;
    const unsigned grid = unsigned(N) * unsigned(HB);
    if (gys != nullptr)
      bn_pool_bwd_k3s2_kernel<true><<<grid, threads, 0, st>>>(
          reinterpret_cast<const float4*>(g_pool), reinterpret_cast<const uint32_t*>(idx),
          reinterpret_cast<const float4*>(y), reinterpret_cast<const float4*>(consts_ws), H, W, C4, Ho, Wo, HB, WB,
          nullptr, amax_scratch, reinterpret_cast<uint2*>(gys));
    else
      bn_pool_bwd_k3s2_kernel<false><<<grid, threads, 0, st>>>(
          reinterpret_cast<const float4*>(g_pool), reinterpret_cast<const uint32_t*>(idx),
          reinterpret_cast<const float4*>(y), reinterpret_cast<const float4*>(consts_ws), H, W, C4, Ho, Wo, HB, WB,
          reinterpret_cast<float4*>(gy), nullptr, nullptr);
    return check_launch("bn_pool_bwd_k3s2_kernel");
  }
  if (gys != nullptr)
    bn_pool_bwd_kernel<true><<<bn_grid(total, C4), kBnThreads, 0, st>>>(
        reinterpret_cast<const float4*>(g_pool), reinterpret_cast<const uint32_t*>(idx),
        reinterpret_cast<const float4*>(y), reinterpret_cast<const float4*>(consts_ws), N, H, W, C4, Ho, Wo, k,
        stride, pad, total, nullptr, amax_scratch, reinterpret_cast<uint2*>(gys));
  else
    bn_pool_bwd_kernel<false><<<bn_grid(total, C4), kBnThreads, 0, st>>>(
        reinterpret_cast<const float4*>(g_pool), reinterpret_cast<const uint32_t*>(idx),
        reinterpret_cast<const float4*>(y), reinterpret_cast<const float4*>(consts_ws), N, H, W, C4, Ho, Wo, k,
        stride, pad, total, reinterpret_cast<float4*>(gy), nullptr, nullptr);
  return check_launch("bn_pool_bwd_kernel");
}
