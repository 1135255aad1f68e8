// Memory-bound training kernels for sm_100a (HBM3e-bound: 128-bit vector accesses, one pass where
// possible, fp32 statistics / accumulation).  These replace the XLA loop/input fusions the reference
// relies on (SURVEY §2.H K10: LayerNorm, GELU, loss, gradient accumulation; K11: optimizer update).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "launch.cuh"

namespace {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return u;
}
__device__ __forceinline__ float tanh_fast(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x));
  return t;
}

// programmatic dependent launch (launch.cuh): every kernel below is launched through tepd::launch and therefore waits for
// its predecessor here, before its first global access
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------ LayerNorm
// One warp per row; each lane owns 8-element vectors at columns (i*32 + lane)*8.
template <int MAXV>  // max vectors per lane (C <= MAXV*256)
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const bf16* __restrict__ x, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, bf16* __restrict__ y,
                                                           float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                           int rows, int C, float eps) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  pdl_wait();
  if (row >= rows) return;
  const int nvec = C >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * C);
  float v[MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = i * 32 + lane;
    if (vi < nvec) {
      uint4 u = __ldg(xr + vi);
      unpack8(u, v[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[i][j];
    }
  }
  const float mean = warp_sum(s) / C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = i * 32 + lane;
    if (vi < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float d = v[i][j] - mean;
        q += d * d;
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / C + eps);
  uint4* yr = reinterpret_cast<uint4*>(y + (size_t)row * C);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = i * 32 + lane;
    if (vi < nvec) {
      const float4* g = reinterpret_cast<const float4*>(gamma + vi * 8);
      const float4* b = reinterpret_cast<const float4*>(beta + vi * 8);
      float4 g0 = __ldg(g), g1 = __ldg(g + 1), b0 = __ldg(b), b1 = __ldg(b + 1);
      float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * gg[j] + bb[j];
      yr[vi] = pack8(o);
    }
  }
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  pdl_trigger();
}

// Backward: dx per row (one warp per row, grid-strided); dgamma / dbeta are accumulated in per-warp SHARED-memory
// rows (no atomics inside the CTA, no 64-register accumulator arrays => 3 CTAs/SM keep enough loads in flight to
// approach HBM bandwidth), reduced across the 8 warps at the end and added (fp32 red) to the gradient buffers.
// Optional dres: fused residual-stream gradient add (dx_total = dx + dres).
// WARPS = 8: 256-thread CTAs, 3 per SM (64 KB of accumulator rows each); WARPS = 16: one 512-thread CTA per SM (128 KB) --
// a third of the CTAs, hence a third of the global atomics on the 2 * C gradient words (TEPDIST_LN_BWD_WARPS selects).
template <int MAXV, int WARPS>
__global__ void __launch_bounds__(32 * WARPS, (MAXV <= 4 && WARPS == 8) ? 3 : 1) layernorm_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ mean_in,
                                                           const float* __restrict__ rstd_in, bf16* __restrict__ dx,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                           const bf16* __restrict__ dres, int rows, int C) {
  extern __shared__ float red[];  // [2][WARPS][C]: dgamma rows then dbeta rows, one per warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = C >> 3;
  float* my_dg = red + (size_t)warp * C;
  float* my_db = red + (size_t)(WARPS + warp) * C;
  for (int c = lane; c < C; c += 32) { my_dg[c] = 0.f; my_db[c] = 0.f; }
  __syncwarp();
  pdl_wait();
  for (int row = blockIdx.x * WARPS + warp; row < rows; row += gridDim.x * WARPS) {
    const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * C);
    const uint4* dyr = reinterpret_cast<const uint4*>(dy + (size_t)row * C);
    const float mean = mean_in[row], rstd = rstd_in[row];
    uint4 xu[MAXV], du[MAXV];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {   // all loads of the row first: 2*MAXV independent 16-byte requests per lane
      const int vi = i * 32 + lane;
      if (vi < nvec) { xu[i] = __ldg(xr + vi); du[i] = __ldg(dyr + vi); }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = i * 32 + lane;
      if (vi < nvec) {
        float xv[8], dv[8];
        unpack8(xu[i], xv);
        unpack8(du[i], dv);
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8) + 1);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        float4* pg = reinterpret_cast<float4*>(my_dg + vi * 8);
        float4* pb = reinterpret_cast<float4*>(my_db + vi * 8);
        float4 a0 = pg[0], a1 = pg[1], b0 = pb[0], b1 = pb[1];
        float ag[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float ab[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (xv[j] - mean) * rstd;
          const float g = dv[j] * gg[j];
          s1 += g;
          s2 += g * xh;
          ag[j] += dv[j] * xh;
          ab[j] += dv[j];
        }
        pg[0] = make_float4(ag[0], ag[1], ag[2], ag[3]); pg[1] = make_float4(ag[4], ag[5], ag[6], ag[7]);
        pb[0] = make_float4(ab[0], ab[1], ab[2], ab[3]); pb[1] = make_float4(ab[4], ab[5], ab[6], ab[7]);
      }
    }
    s1 = warp_sum(s1) / C;
    s2 = warp_sum(s2) / C;
    uint4* dxr = reinterpret_cast<uint4*>(dx + (size_t)row * C);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = i * 32 + lane;
      if (vi < nvec) {
        float xv[8], dv[8], o[8];
        unpack8(xu[i], xv);
        unpack8(du[i], dv);
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8) + 1);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = rstd * (dv[j] * gg[j] - s1 - (xv[j] - mean) * rstd * s2);
        if (dres) {  // fused residual-stream gradient add
          float rr[8];
          unpack8(__ldg(reinterpret_cast<const uint4*>(dres + (size_t)row * C) + vi), rr);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] += rr[j];
        }
        dxr[vi] = pack8(o);
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 32 * WARPS) {
    float sg = 0.f, sb = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) { sg += red[(size_t)w * C + c]; sb += red[(size_t)(WARPS + w) * C + c]; }
    atomicAdd(dgamma + c, sg);
    atomicAdd(dbeta + c, sb);
  }
}

// ------------------------------------------------------------------ GELU (tanh form, GPT-2)
__device__ __forceinline__ float gelu_f(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  return 0.5f * x * (1.f + tanh_fast(k0 * (x + k1 * x * x * x)));
}
__device__ __forceinline__ float gelu_grad_f(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float t = tanh_fast(k0 * (x + k1 * x * x * x));
  float dt = (1.f - t * t) * k0 * (1.f + 3.f * k1 * x * x);
  return 0.5f * (1.f + t) + 0.5f * x * dt;
}
__global__ void gelu_fwd_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, size_t nvec) {
  pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    float f[8];
    unpack8(__ldg(x + i), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = gelu_f(f[j]);
    y[i] = pack8(f);
  }
}
// dx = dy * gelu'(x);  optionally also accumulates the column sums of dx? (no: bias grad handled by colsum)
__global__ void gelu_bwd_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ x, uint4* __restrict__ dx,
                                size_t nvec) {
  pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    float f[8], d[8];
    unpack8(__ldg(x + i), f);
    unpack8(__ldg(dy + i), d);
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] *= gelu_grad_f(f[j]);
    dx[i] = pack8(d);
  }
}

// ------------------------------------------------------------------ BatchNorm (training mode) on NHWC rows
// x is [rows = N*H*W, C] (channels_last memory).  Two passes each way, both column-parallel like colsum:
//   forward : bn_reduce2 accumulates sum(x) and sum(x^2) per channel (fp32 atomics over row strips), bn_fwd_apply turns
//             them into mean / rstd and writes y = (x - mean) * rstd * gamma + beta (+ ReLU);
//   backward: bn_reduce2 with dy accumulates sum(dy) and sum(dy * xhat), bn_bwd_apply writes
//             dx = gamma * rstd * (dy - mean(dy) - xhat * mean(dy * xhat)).
// MODE 0: (x, x^2); MODE 1: (dy, dy * xhat) with xhat recomputed from x, mean, rstd.
template <int MODE>
__global__ void __launch_bounds__(256) bn_reduce2_kernel(const bf16* __restrict__ a, const bf16* __restrict__ x,
                                                        const float* __restrict__ mean, const float* __restrict__ rstd,
                                                        float* __restrict__ out0, float* __restrict__ out1, int rows, int C,
                                                        int rows_per_block) {
  __shared__ float red[2][8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = blockIdx.x * 256 + lane * 8;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(rows, r0 + rows_per_block);
  float s0[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s1[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  pdl_wait();
  if (col0 < C) {
    float mu[8], rs[8];
    if (MODE == 1) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { mu[j] = mean[col0 + j]; rs[j] = rstd[col0 + j]; }
    }
    for (int r = r0 + warp; r < r1; r += 8) {
      float f[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(a + (size_t)r * C + col0)), f);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { s0[j] += f[j]; s1[j] += f[j] * f[j]; }
      } else {
        float xv[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(x + (size_t)r * C + col0)), xv);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s0[j] += f[j]; s1[j] += f[j] * (xv[j] - mu[j]) * rs[j]; }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) { red[0][warp][lane * 8 + j] = s0[j]; red[1][warp][lane * 8 + j] = s1[j]; }
  __syncthreads();
  const int c = threadIdx.x;
  if (blockIdx.x * 256 + c < C) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { t0 += red[0][w][c]; t1 += red[1][w][c]; }
    atomicAdd(out0 + blockIdx.x * 256 + c, t0);
    atomicAdd(out1 + blockIdx.x * 256 + c, t1);
  }
}

// sums = [sum(x), sum(x^2)] -> mean, rstd (written by block row 0) and y
__global__ void __launch_bounds__(256) bn_fwd_apply_kernel(const bf16* __restrict__ x, const float* __restrict__ sum,
                                                          const float* __restrict__ sumsq, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, bf16* __restrict__ y,
                                                          float* __restrict__ mean_out, float* __restrict__ rstd_out, int rows,
                                                          int C, float eps, int relu, float count) {
  pdl_wait();
  const int cv = C >> 3;
  const float inv = 1.f / count;     // count = rows of the GLOBAL batch (rows of every shard when the batch is split)
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)rows * cv; i += (size_t)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % cv) * 8;
    float f[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x) + i), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float mu = sum[c0 + j] * inv;
      const float var = fmaxf(sumsq[c0 + j] * inv - mu * mu, 0.f);
      const float rs = rsqrtf(var + eps);
      float v = (f[j] - mu) * rs * gamma[c0 + j] + beta[c0 + j];
      o[j] = relu ? fmaxf(v, 0.f) : v;
      if (i < (size_t)cv) { mean_out[c0 + j] = mu; rstd_out[c0 + j] = rs; }
    }
    reinterpret_cast<uint4*>(y)[i] = pack8(o);
  }
}

__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                          const float* __restrict__ gamma, const float* __restrict__ mean,
                                                          const float* __restrict__ rstd, const float* __restrict__ sum_dy,
                                                          const float* __restrict__ sum_dyxh, bf16* __restrict__ dx, int rows, int C,
                                                          float count) {
  pdl_wait();
  const int cv = C >> 3;
  const float inv = 1.f / count;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)rows * cv; i += (size_t)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % cv) * 8;
    float d[8], f[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy) + i), d);
    unpack8(__ldg(reinterpret_cast<const uint4*>(x) + i), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float rs = rstd[c0 + j];
      const float xh = (f[j] - mean[c0 + j]) * rs;
      o[j] = gamma[c0 + j] * rs * (d[j] - sum_dy[c0 + j] * inv - xh * sum_dyxh[c0 + j] * inv);
    }
    reinterpret_cast<uint4*>(dx)[i] = pack8(o);
  }
}

// ------------------------------------------------------------------ column sum (bias gradients)
// out[c] += sum_r in[r, c];  block handles 256 columns (32 lanes x 8) x a strip of rows.
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ in, float* __restrict__ out, int rows, int C,
                                                    int rows_per_block) {
  __shared__ float red[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = blockIdx.x * 256 + lane * 8;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(rows, r0 + rows_per_block);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  pdl_wait();
  if (col0 < C) {
    int r = r0 + warp;
    for (; r + 24 < r1; r += 32) {   // 4 rows in flight per lane
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) u[k] = __ldg(reinterpret_cast<const uint4*>(in + (size_t)(r + 8 * k) * C + col0));
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float f[8];
        unpack8(u[k], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
    for (; r < r1; r += 8) {
      float f[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(in + (size_t)r * C + col0)), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[warp][lane * 8 + j] = acc[j];
  __syncthreads();
  const int c = threadIdx.x;
  if (blockIdx.x * 256 + c < C) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][c];
    atomicAdd(out + blockIdx.x * 256 + c, s);
  }
}

// ------------------------------------------------------------------ embedding
__global__ void embedding_fwd_kernel(const int* __restrict__ tok, const bf16* __restrict__ wte, const bf16* __restrict__ wpe,
                                     bf16* __restrict__ out, int T, int S, int C) {
  const int nvec = C >> 3;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)T * nvec;
       i += (size_t)gridDim.x * blockDim.x) {
    const int t = i / nvec, v = i % nvec;
    const int id = tok[t], pos = t % S;
    float a[8], b[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(wte + (size_t)id * C) + v), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(wpe + (size_t)pos * C) + v), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += b[j];
    reinterpret_cast<uint4*>(out + (size_t)t * C)[v] = pack8(a);
  }
}
__global__ void embedding_bwd_kernel(const int* __restrict__ tok, const bf16* __restrict__ dout, float* __restrict__ dwte,
                                     float* __restrict__ dwpe, int T, int S, int C) {
  const int nvec = C >> 3;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)T * nvec;
       i += (size_t)gridDim.x * blockDim.x) {
    const int t = i / nvec, v = i % nvec;
    const int id = tok[t], pos = t % S;
    float d[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(dout + (size_t)t * C) + v), d);
    float* pe = dwte + (size_t)id * C + v * 8;
    float* pp = dwpe + (size_t)pos * C + v * 8;
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(pe), "f"(d[0]), "f"(d[1]), "f"(d[2]), "f"(d[3]) : "memory");
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(pe + 4), "f"(d[4]), "f"(d[5]), "f"(d[6]), "f"(d[7]) : "memory");
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(pp), "f"(d[0]), "f"(d[1]), "f"(d[2]), "f"(d[3]) : "memory");
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(pp + 4), "f"(d[4]), "f"(d[5]), "f"(d[6]), "f"(d[7]) : "memory");
  }
}

// ------------------------------------------------------------------ softmax cross-entropy (fused fwd+bwd)
// One block per row.  logits [T, Vp] bf16 (Vp = padded vocab, columns >= V are ignored and get zero
// gradient).  Writes per-row loss and overwrites logits with dlogits = (softmax - onehot) * gscale.
__global__ void __launch_bounds__(512) xent_fwd_bwd_kernel(bf16* __restrict__ logits, const int* __restrict__ labels,
                                                          float* __restrict__ loss_rows, float* __restrict__ loss_sum,
                                                          int V, int Vp, float gscale) {
  __shared__ float sred[16];
  __shared__ float sbc;
  const int row = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint4* lr = reinterpret_cast<uint4*>(logits + (size_t)row * Vp);
  const int nvec = Vp >> 3;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < nvec; i += 512) {
    float f[8];
    unpack8(lr[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (i * 8 + j < V) mx = fmaxf(mx, f[j]);
  }
  mx = warp_max(mx);
  if (lane == 0) sred[warp] = mx;
  __syncthreads();
  if (warp == 0) {
    float m = lane < 16 ? sred[lane] : -INFINITY;
    m = warp_max(m);
    if (lane == 0) sbc = m;
  }
  __syncthreads();
  mx = sbc;
  float se = 0.f;
  for (int i = threadIdx.x; i < nvec; i += 512) {
    float f[8];
    unpack8(lr[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (i * 8 + j < V) se += __expf(f[j] - mx);
  }
  se = warp_sum(se);
  __syncthreads();
  if (lane == 0) sred[warp] = se;
  __syncthreads();
  if (warp == 0) {
    float s = lane < 16 ? sred[lane] : 0.f;
    s = warp_sum(s);
    if (lane == 0) sbc = s;
  }
  __syncthreads();
  se = sbc;
  const int lab = labels[row];
  const float inv = 1.f / se;
  for (int i = threadIdx.x; i < nvec; i += 512) {
    float f[8];
    unpack8(lr[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = i * 8 + j;
      float p = c < V ? __expf(f[j] - mx) * inv : 0.f;
      if (c == lab) {
        float l = -(f[j] - mx - __logf(se));
        loss_rows[row] = l;
        atomicAdd(loss_sum, l * gscale);
        p -= 1.f;
      }
      f[j] = p * gscale;
    }
    lr[i] = pack8(f);
  }
}

// ------------------------------------------------------------------ fused AdamW over flat buffers
// master fp32 params, fp32 grads (already summed/averaged), fp32 m/v; writes the bf16 compute copy.
// wd_mask: per-"segment" weight decay is encoded by the caller splitting the flat buffer into a decayed
// prefix [0, n_decay) and a non-decayed suffix.
__device__ __forceinline__ void adamw_one(float& p, float g, float& m, float& v, float lr, float beta1, float beta2,
                                          float eps, float decay, float bc1, float bc2) {
  m = beta1 * m + (1.f - beta1) * g;
  v = beta2 * v + (1.f - beta2) * g * g;
  const float mh = m / bc1, vh = v / bc2;
  p -= lr * (mh / (sqrtf(vh) + eps) + decay * p);
}
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, bf16* __restrict__ p_bf16, size_t n, size_t n_decay, float lr,
                             float beta1, float beta2, float eps, float wd, float bc1, float bc2, float gscale,
                             const float* __restrict__ hyper) {
  // hyper (device, optional): {lr, bc1, bc2, gscale} so a captured CUDA graph sees per-step values
  if (hyper) { lr = hyper[0]; bc1 = hyper[1]; bc2 = hyper[2]; gscale = hyper[3]; }
  const size_t nvec = n >> 2;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float pa[4] = {pp.x, pp.y, pp.z, pp.w}, ga[4] = {gg.x, gg.y, gg.z, gg.w};
    float ma[4] = {mm.x, mm.y, mm.z, mm.w}, va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      adamw_one(pa[j], ga[j] * gscale, ma[j], va[j], lr, beta1, beta2, eps, (i * 4 + j < n_decay) ? wd : 0.f, bc1, bc2);
    reinterpret_cast<float4*>(p)[i] = make_float4(pa[0], pa[1], pa[2], pa[3]);
    reinterpret_cast<float4*>(m)[i] = make_float4(ma[0], ma[1], ma[2], ma[3]);
    reinterpret_cast<float4*>(v)[i] = make_float4(va[0], va[1], va[2], va[3]);
    if (p_bf16) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(pa[0], pa[1]), hi = __floats2bfloat162_rn(pa[2], pa[3]);
      uint2 u;
      u.x = *reinterpret_cast<uint32_t*>(&lo);
      u.y = *reinterpret_cast<uint32_t*>(&hi);
      reinterpret_cast<uint2*>(p_bf16)[i] = u;
    }
  }
  // scalar tail (n not a multiple of 4)
  for (size_t i = (nvec << 2) + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float pa = p[i], ma = m[i], va = v[i];
    adamw_one(pa, g[i] * gscale, ma, va, lr, beta1, beta2, eps, (i < n_decay) ? wd : 0.f, bc1, bc2);
    p[i] = pa; m[i] = ma; v[i] = va;
    if (p_bf16) p_bf16[i] = __float2bfloat16(pa);
  }
}

// SGD (smoke examples use plain SGD).
__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, bf16* __restrict__ p_bf16, size_t n,
                           float lr, float gscale) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float x = p[i] - lr * g[i] * gscale;
    p[i] = x;
    if (p_bf16) p_bf16[i] = __float2bfloat16(x);
  }
}

// acc += g  (gradient accumulation "GA" task on fp32 buffers); cast helper.
__global__ void axpy_f32_kernel(float* __restrict__ acc, const float* __restrict__ g, size_t n, float a) {
  const size_t nvec = n >> 2;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    float4 x = reinterpret_cast<float4*>(acc)[i];
    float4 y = reinterpret_cast<const float4*>(g)[i];
    x.x += a * y.x; x.y += a * y.y; x.z += a * y.z; x.w += a * y.w;
    reinterpret_cast<float4*>(acc)[i] = x;
  }
}
__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16(in[i]);
}
// ---- dense bf16 elementwise (conv nets: ReLU, ReLU backward, residual add); MODE 0: relu(a), 1: a * (b > 0), 2: a + b
template <int MODE>
__global__ void __launch_bounds__(256) ew_bf16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out,
                                                      size_t nvec) {
  pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    float x[8], y[8], o[8];
    unpack8(__ldg(a + i), x);
    if (MODE != 0) unpack8(__ldg(b + i), y);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = MODE == 0 ? fmaxf(x[j], 0.f) : (MODE == 1 ? (y[j] > 0.f ? x[j] : 0.f) : x[j] + y[j]);
    out[i] = pack8(o);
  }
}
// 8 elements per thread: two 16-byte loads, one 16-byte store (pointers 32 / 16-byte aligned, n % 8 == 0)
__global__ void __launch_bounds__(256) cast_f32_bf16_vec_kernel(const float4* __restrict__ in, uint4* __restrict__ out, size_t nvec) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    const float4 a = __ldg(in + 2 * i), b = __ldg(in + 2 * i + 1);
    uint4 u;
    __nv_bfloat162 h;
    h = __floats2bfloat162_rn(a.x, a.y); u.x = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(a.z, a.w); u.y = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(b.x, b.y); u.z = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(b.z, b.w); u.w = *reinterpret_cast<uint32_t*>(&h);
    out[i] = u;
  }
}

// ---- ring (context-parallel) attention helpers.  Layouts: o / dq [B,L,H,D], lse [B,H,L], qkv-like [B,L,H,3,D], kv-like [B,L,H,2,D];
// D % 8 == 0; one thread per 8 consecutive d.
// merge: (o_acc, lse_in) <- log-sum-exp merge with one block's (o_j, lse_j); lse written to lse_out (ping-pong: every thread of a
// row reads lse_in).  first != 0: plain initialisation.
__global__ void __launch_bounds__(256) attn_merge_kernel(float* __restrict__ o_acc, const float* __restrict__ lse_in,
                                                         float* __restrict__ lse_out, const bf16* __restrict__ o_j,
                                                         const float* __restrict__ lse_j, int B, int L, int H, int D, int first) {
  const int dv = D / 8;
  const size_t nvec = (size_t)B * L * H * dv;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i / dv;                     // (b, l, h)
    const int h = (int)(row % H), l = (int)((row / H) % L), b = (int)(row / ((size_t)H * L));
    const size_t li = ((size_t)b * H + h) * L + l;
    float x[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(o_j) + i), x);
    float4* oa = reinterpret_cast<float4*>(o_acc) + 2 * i;
    const float lj = __ldg(lse_j + li);
    if (first) {
      oa[0] = make_float4(x[0], x[1], x[2], x[3]);
      oa[1] = make_float4(x[4], x[5], x[6], x[7]);
      if (i % dv == 0) lse_out[li] = lj;
      continue;
    }
    const float la = __ldg(lse_in + li);
    const float mx = fmaxf(la, lj);
    // both partials empty (document masking: no key of either block is visible to the row): stay at o = 0, lse = -inf
    const bool empty = mx == -INFINITY;
    const float nw = empty ? -INFINITY : mx + __logf(__expf(la - mx) + __expf(lj - mx));
    const float wa = empty ? 0.f : __expf(la - nw), wj = empty ? 0.f : __expf(lj - nw);
    float4 a0 = oa[0], a1 = oa[1];
    a0.x = a0.x * wa + x[0] * wj; a0.y = a0.y * wa + x[1] * wj; a0.z = a0.z * wa + x[2] * wj; a0.w = a0.w * wa + x[3] * wj;
    a1.x = a1.x * wa + x[4] * wj; a1.y = a1.y * wa + x[5] * wj; a1.z = a1.z * wa + x[6] * wj; a1.w = a1.w * wa + x[7] * wj;
    oa[0] = a0; oa[1] = a1;
    if (i % dv == 0) lse_out[li] = nw;
  }
}
// accum: dq_acc [B,L,H,D] += part[..,0,:];  kv_acc [B,L,H,2,D] += part[..,1:3,:]   (part = one block's bf16 dq / dk / dv)
// pack (PACK = 1): the inverse at the end of the ring: part[..,0,:] = bf16(dq_acc), part[..,1:3,:] = bf16(kv_acc)
template <int PACK>
__global__ void __launch_bounds__(256) attn_ring_accum_kernel(float* __restrict__ dq_acc, float* __restrict__ kv_acc, bf16* __restrict__ part,
                                                              size_t rows, int D) {
  const int dv = D / 8;
  const size_t nvec = rows * 3 * dv;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % dv), slot = (int)((i / dv) % 3);
    const size_t row = i / ((size_t)3 * dv);
    float* dst = slot == 0 ? dq_acc + (row * D + (size_t)c * 8) : kv_acc + ((row * 2 + (slot - 1)) * D + (size_t)c * 8);
    float4* d4 = reinterpret_cast<float4*>(dst);
    if (PACK) {
      const float4 a0 = d4[0], a1 = d4[1];
      float o[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      reinterpret_cast<uint4*>(part)[i] = pack8(o);
    } else {
      float x[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(part) + i), x);
      float4 a0 = d4[0], a1 = d4[1];
      a0.x += x[0]; a0.y += x[1]; a0.z += x[2]; a0.w += x[3];
      a1.x += x[4]; a1.y += x[5]; a1.z += x[6]; a1.w += x[7];
      d4[0] = a0; d4[1] = a1;
    }
  }
}

inline int grid_for(size_t work, int threads) {
  size_t b = (work + threads - 1) / threads;
  size_t cap = 148 * 8;
  return (int)(b < cap ? (b ? b : 1) : cap);
}

}  // namespace

#define CS(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int tepd_layernorm_fwd(const void* x, const void* gamma, const void* beta, void* y, void* mean, void* rstd,
                                  int rows, int C, float eps, void* stream) {
  if (C % 8 || C > 4096) return -2;
  dim3 grid((rows + 7) / 8);
#define LN_FWD(MV) return (int)tepd::launch(layernorm_fwd_kernel<MV>, grid, dim3(256), 0, CS(stream), (const bf16*)x, (const float*)gamma, (const float*)beta, (bf16*)y, (float*)mean, (float*)rstd, rows, C, eps)
  if (C <= 1024) LN_FWD(4); else if (C <= 2048) LN_FWD(8); else LN_FWD(16);
#undef LN_FWD
}

extern "C" int tepd_layernorm_bwd(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd,
                                  void* dx, void* dgamma, void* dbeta, const void* dres, int rows, int C, void* stream) {
  if (C % 8 || C > 2048) return -2;
  int grid = 148 * 3;
  static int warps = 0;
  if (warps == 0) {
    const char* e = getenv("TEPDIST_LN_BWD_WARPS");
    warps = (e && atoi(e) == 8) ? 8 : 16;      // measured in situ (GPT-2 345M, 49 launches): 15.6 us (16 warps, 148 CTAs) vs 17.2 us (8 warps, 444 CTAs)
  }
  if (warps == 16 && C > 1024) warps = 8;      // (2 * 16 * C floats must fit one CTA's shared memory)
  if (warps == 16) grid = 148;
  if (grid > (rows + warps - 1) / warps) grid = (rows + warps - 1) / warps;
  size_t smem = (size_t)2 * warps * C * sizeof(float);
#define LN_BWD(MV, W)                                                                                       \
  {                                                                                                         \
    static bool cfg = false;                                                                                \
    if (!cfg) { cudaFuncSetAttribute(layernorm_bwd_kernel<MV, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * W * 2048 * 4 > 200 * 1024 ? 200 * 1024 : 2 * W * 2048 * 4); cfg = true; } \
    return (int)tepd::launch(layernorm_bwd_kernel<MV, W>, dim3(grid), dim3(32 * W), smem, CS(stream), (const bf16*)dy, (const bf16*)x, (const float*)gamma, (const float*)mean, (const float*)rstd, (bf16*)dx, (float*)dgamma, (float*)dbeta, (const bf16*)dres, rows, C); \
  }
  if (C <= 1024) { if (warps == 16) LN_BWD(4, 16) else LN_BWD(4, 8) } else LN_BWD(8, 8)
#undef LN_BWD
}

extern "C" int tepd_gelu_fwd(const void* x, void* y, long long n, void* stream) {
  if (n % 8) return -2;
  return (int)tepd::launch(gelu_fwd_kernel, dim3(grid_for(n / 8, 256)), dim3(256), 0, CS(stream), (const uint4*)x, (uint4*)y, (size_t)(n / 8));
}
extern "C" int tepd_gelu_bwd(const void* dy, const void* x, void* dx, long long n, void* stream) {
  if (n % 8) return -2;
  return (int)tepd::launch(gelu_bwd_kernel, dim3(grid_for(n / 8, 256)), dim3(256), 0, CS(stream), (const uint4*)dy, (const uint4*)x, (uint4*)dx, (size_t)(n / 8));
}
extern "C" int tepd_colsum(const void* in, void* out, int rows, int C, void* stream) {
  if (C % 8) return -2;
  int rpb = 64;
  dim3 grid((C + 255) / 256, (rows + rpb - 1) / rpb);
  return (int)tepd::launch(colsum_kernel, grid, dim3(256), 0, CS(stream), (const bf16*)in, (float*)out, rows, C, rpb);
  return (int)cudaGetLastError();
}
extern "C" int tepd_embedding_fwd(const void* tok, const void* wte, const void* wpe, void* out, int T, int S, int C,
                                  void* stream) {
  if (C % 8) return -2;
  embedding_fwd_kernel<<<grid_for((size_t)T * C / 8, 256), 256, 0, CS(stream)>>>((const int*)tok, (const bf16*)wte, (const bf16*)wpe, (bf16*)out, T, S, C);
  return (int)cudaGetLastError();
}
extern "C" int tepd_embedding_bwd(const void* tok, const void* dout, void* dwte, void* dwpe, int T, int S, int C,
                                  void* stream) {
  if (C % 8) return -2;
  embedding_bwd_kernel<<<grid_for((size_t)T * C / 8, 256), 256, 0, CS(stream)>>>((const int*)tok, (const bf16*)dout, (float*)dwte, (float*)dwpe, T, S, C);
  return (int)cudaGetLastError();
}
extern "C" int tepd_xent_fwd_bwd(void* logits, const void* labels, void* loss_rows, void* loss_sum, int T, int V, int Vp,
                                 float gscale, void* stream) {
  if (Vp % 8) return -2;
  xent_fwd_bwd_kernel<<<T, 512, 0, CS(stream)>>>((bf16*)logits, (const int*)labels, (float*)loss_rows, (float*)loss_sum, V, Vp, gscale);
  return (int)cudaGetLastError();
}
extern "C" int tepd_adamw(void* p, const void* g, void* m, void* v, void* p_bf16, long long n, long long n_decay, float lr,
                          float beta1, float beta2, float eps, float wd, float bc1, float bc2, float gscale,
                          const void* hyper, void* stream) {
  if ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15) return -2;
  if (p_bf16 && (reinterpret_cast<uintptr_t>(p_bf16) & 7)) return -3;
  adamw_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, CS(stream)>>>((float*)p, (const float*)g, (float*)m, (float*)v, (bf16*)p_bf16, n, n_decay, lr, beta1, beta2, eps, wd, bc1, bc2, gscale, (const float*)hyper);
  return (int)cudaGetLastError();
}
extern "C" int tepd_sgd(void* p, const void* g, void* p_bf16, long long n, float lr, float gscale, void* stream) {
  sgd_kernel<<<grid_for(n, 256), 256, 0, CS(stream)>>>((float*)p, (const float*)g, (bf16*)p_bf16, n, lr, gscale);
  return (int)cudaGetLastError();
}
extern "C" int tepd_axpy_f32(void* acc, const void* g, long long n, float a, void* stream) {
  if (n % 4) return -2;
  axpy_f32_kernel<<<grid_for(n / 4, 256), 256, 0, CS(stream)>>>((float*)acc, (const float*)g, n, a);
  return (int)cudaGetLastError();
}
// out = relu(a) (mode 0) | a * (b > 0) (mode 1: ReLU backward with b = the forward OUTPUT) | a + b (mode 2); n % 8 == 0, 16-byte aligned
extern "C" int tepd_ew_bf16(const void* a, const void* b, void* out, long long n, int mode, void* stream) {
  if (n % 8 || ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(b)) & 15)) return -2;
  const size_t nvec = (size_t)(n / 8);
  dim3 grid(grid_for(nvec, 256));
  if (mode == 0) return (int)tepd::launch(ew_bf16_kernel<0>, grid, dim3(256), 0, CS(stream), (const uint4*)a, (const uint4*)b, (uint4*)out, nvec);
  if (mode == 1) return (int)tepd::launch(ew_bf16_kernel<1>, grid, dim3(256), 0, CS(stream), (const uint4*)a, (const uint4*)b, (uint4*)out, nvec);
  return (int)tepd::launch(ew_bf16_kernel<2>, grid, dim3(256), 0, CS(stream), (const uint4*)a, (const uint4*)b, (uint4*)out, nvec);
}
extern "C" int tepd_attn_merge(void* o_acc, const void* lse_in, void* lse_out, const void* o_j, const void* lse_j, int B, int L, int H,
                               int D, int first, void* stream) {
  if (D % 8 || ((reinterpret_cast<uintptr_t>(o_acc) | reinterpret_cast<uintptr_t>(o_j)) & 15)) return -2;
  attn_merge_kernel<<<grid_for((size_t)B * L * H * (D / 8), 256), 256, 0, CS(stream)>>>((float*)o_acc, (const float*)lse_in, (float*)lse_out,
                                                                                      (const bf16*)o_j, (const float*)lse_j, B, L, H, D, first);
  return (int)cudaGetLastError();
}
extern "C" int tepd_attn_ring_accum(void* dq_acc, void* kv_acc, void* part, long long rows, int D, int pack, void* stream) {
  if (D % 8 || ((reinterpret_cast<uintptr_t>(dq_acc) | reinterpret_cast<uintptr_t>(kv_acc) | reinterpret_cast<uintptr_t>(part)) & 15)) return -2;
  const int grid = grid_for((size_t)rows * 3 * (D / 8), 256);
  if (pack) attn_ring_accum_kernel<1><<<grid, 256, 0, CS(stream)>>>((float*)dq_acc, (float*)kv_acc, (bf16*)part, (size_t)rows, D);
  else attn_ring_accum_kernel<0><<<grid, 256, 0, CS(stream)>>>((float*)dq_acc, (float*)kv_acc, (bf16*)part, (size_t)rows, D);
  return (int)cudaGetLastError();
}
extern "C" int tepd_cast_f32_bf16(const void* in, void* out, long long n, void* stream) {
  if (n % 8 == 0 && (reinterpret_cast<uintptr_t>(in) & 31) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0)
    cast_f32_bf16_vec_kernel<<<grid_for(n / 8, 256), 256, 0, CS(stream)>>>((const float4*)in, (uint4*)out, (size_t)(n / 8));
  else
    cast_f32_bf16_kernel<<<grid_for(n, 256), 256, 0, CS(stream)>>>((const float*)in, (bf16*)out, n);
  return (int)cudaGetLastError();
}

// ---- BatchNorm NHWC.  ws: fp32 [2, C] scratch, zeroed by the caller (sum / sumsq, or sum(dy) / sum(dy*xhat) which the
// backward ALSO adds into dbeta / dgamma: the caller points ws at zero-filled temporaries and accumulates them itself).
extern "C" int tepd_bn_fwd_nhwc(const void* x, const void* gamma, const void* beta, void* y, void* mean, void* rstd, void* ws,
                                int rows, int C, float eps, int relu, void* stream) {
  if (C % 8) return -2;
  const int rpb = 128;
  dim3 grid((C + 255) / 256, (rows + rpb - 1) / rpb);
  float* w = (float*)ws;
  cudaError_t e = tepd::launch(bn_reduce2_kernel<0>, grid, dim3(256), 0, CS(stream), (const bf16*)x, (const bf16*)nullptr,
                               (const float*)nullptr, (const float*)nullptr, w, w + C, rows, C, rpb);
  if (e != cudaSuccess) return (int)e;
  return (int)tepd::launch(bn_fwd_apply_kernel, dim3(grid_for((size_t)rows * C / 8, 256)), dim3(256), 0, CS(stream), (const bf16*)x,
                           (const float*)w, (const float*)(w + C), (const float*)gamma, (const float*)beta, (bf16*)y, (float*)mean,
                           (float*)rstd, rows, C, eps, relu, (float)rows);
}
extern "C" int tepd_bn_bwd_nhwc(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, void* dx,
                                void* ws, int rows, int C, void* stream) {
  if (C % 8) return -2;
  const int rpb = 128;
  dim3 grid((C + 255) / 256, (rows + rpb - 1) / rpb);
  float* w = (float*)ws;
  cudaError_t e = tepd::launch(bn_reduce2_kernel<1>, grid, dim3(256), 0, CS(stream), (const bf16*)dy, (const bf16*)x,
                               (const float*)mean, (const float*)rstd, w, w + C, rows, C, rpb);
  if (e != cudaSuccess) return (int)e;
  return (int)tepd::launch(bn_bwd_apply_kernel, dim3(grid_for((size_t)rows * C / 8, 256)), dim3(256), 0, CS(stream), (const bf16*)dy,
                           (const bf16*)x, (const float*)gamma, (const float*)mean, (const float*)rstd, (const float*)w,
                           (const float*)(w + C), (bf16*)dx, rows, C, (float)rows);
}
// Split-phase BatchNorm for a batch that is split over devices (synchronised BatchNorm): the per-channel sums of the local
// shard are produced by `tepd_bn_reduce_nhwc`, completed across the devices by an all-reduce of the 2 x C words, and consumed
// by the apply halves with the GLOBAL row count.  mode 0: ws = [sum(x), sum(x^2)]; mode 1: ws = [sum(dy), sum(dy * xhat)].
extern "C" int tepd_bn_reduce_nhwc(const void* a, const void* x, const void* mean, const void* rstd, void* ws, int rows, int C, int mode,
                                   void* stream) {
  if (C % 8) return -2;
  const int rpb = 128;
  dim3 grid((C + 255) / 256, (rows + rpb - 1) / rpb);
  float* w = (float*)ws;
  if (mode == 0)
    return (int)tepd::launch(bn_reduce2_kernel<0>, grid, dim3(256), 0, CS(stream), (const bf16*)a, (const bf16*)nullptr,
                             (const float*)nullptr, (const float*)nullptr, w, w + C, rows, C, rpb);
  return (int)tepd::launch(bn_reduce2_kernel<1>, grid, dim3(256), 0, CS(stream), (const bf16*)a, (const bf16*)x, (const float*)mean,
                           (const float*)rstd, w, w + C, rows, C, rpb);
}
extern "C" int tepd_bn_fwd_apply_nhwc(const void* x, const void* ws, const void* gamma, const void* beta, void* y, void* mean, void* rstd,
                                      int rows, int C, float eps, int relu, float count, void* stream) {
  if (C % 8) return -2;
  const float* w = (const float*)ws;
  return (int)tepd::launch(bn_fwd_apply_kernel, dim3(grid_for((size_t)rows * C / 8, 256)), dim3(256), 0, CS(stream), (const bf16*)x, w,
                           w + C, (const float*)gamma, (const float*)beta, (bf16*)y, (float*)mean, (float*)rstd, rows, C, eps, relu, count);
}
extern "C" int tepd_bn_bwd_apply_nhwc(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, const void* ws,
                                      void* dx, int rows, int C, float count, void* stream) {
  if (C % 8) return -2;
  const float* w = (const float*)ws;
  return (int)tepd::launch(bn_bwd_apply_kernel, dim3(grid_for((size_t)rows * C / 8, 256)), dim3(256), 0, CS(stream), (const bf16*)dy,
                           (const bf16*)x, (const float*)gamma, (const float*)mean, (const float*)rstd, w, w + C, (bf16*)dx, rows, C, count);
}
