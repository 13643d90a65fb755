// CLIP-side row kernels: LayerNorm fwd/bwd on the fp32 residual stream, attention softmax fwd/bwd, the
// class-token head (ln_post + proj), the Prompt / spherical-distance loss with its gradient, the optimiser step + clip_z.
#include "kernels.cuh"
#include "launch.cuh"
#include <cfloat>
#include <cmath>
#include <stdexcept>

namespace pxr {
namespace {

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

constexpr int LN_MAX_VEC = 8;  // W <= 1024, W % 128 == 0: each lane owns W/128 float4 vectors of the row

__device__ __forceinline__ void st_half4(act_t* p, float a, float b, float c, float d) {
  __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo);
  u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ float4 ld_half4(const act_t* p) {
  uint2 u = *reinterpret_cast<const uint2*>(p);
  float2 a = __half22float2(*reinterpret_cast<__half2*>(&u.x)), b = __half22float2(*reinterpret_cast<__half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// 4 consecutive elements of a residual-stream row, fp32 (16-byte load) or fp16 (8-byte load)
__device__ __forceinline__ float4 ld_x4(const float* p, int c4) { return reinterpret_cast<const float4*>(p)[c4]; }
__device__ __forceinline__ float4 ld_x4(const act_t* p, int c4) { return ld_half4(p + 4 * c4); }

// one warp per row; vector accesses; x rows are x_stride apart (class-token rows: T * W).  XT = float: the fp32 residual
// stream; XT = act_t: the fp16 one (what the reference's own CUDA path keeps, slip.py:176 / clip.load(..., jit=False).half()).
template <int NV, typename XT>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const XT* __restrict__ x, long long x_stride,
                                                            const float* __restrict__ pos, int T,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, int rows, int W, float eps,
                                                            act_t* __restrict__ y16, float* __restrict__ y32,
                                                            float* __restrict__ stats) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float4 v[NV];
  const XT* xr = x + (size_t)row * x_stride;
  const float4* pr = pos ? reinterpret_cast<const float4*>(pos + (size_t)(row % T) * W) : nullptr;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float4 t = ld_x4(xr, lane + 32 * i);
    if (pr) {
      float4 q = pr[lane + 32 * i];
      t.x += q.x;
      t.y += q.y;
      t.z += q.z;
      t.w += q.w;
    }
    v[i] = t;
    s += (t.x + t.y) + (t.z + t.w);
  }
  const float mean = warp_sum(s) / W;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(q) / W + eps);
  if (lane == 0) {
    stats[2 * row] = mean;
    stats[2 * row + 1] = rstd;
  }
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c4 = lane + 32 * i;
    float4 g = g4[c4], bb = b4[c4];
    float o0 = (v[i].x - mean) * rstd * g.x + bb.x, o1 = (v[i].y - mean) * rstd * g.y + bb.y;
    float o2 = (v[i].z - mean) * rstd * g.z + bb.z, o3 = (v[i].w - mean) * rstd * g.w + bb.w;
    if (y16) st_half4(y16 + (size_t)row * W + 4 * c4, o0, o1, o2, o3);
    if (y32) reinterpret_cast<float4*>(y32 + (size_t)row * W)[c4] = make_float4(o0, o1, o2, o3);
  }
}

// gx == nullptr: the gradient of the residual stream lives in gx16 alone (fp16 stream): accumulate reads it from there
template <int NV, typename XT>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const act_t* __restrict__ dy, const XT* __restrict__ x,
                                                            long long x_stride, const float* __restrict__ pos, int T,
                                                            const float* __restrict__ stats,
                                                            const float* __restrict__ gamma, int rows, int W,
                                                            int accumulate, float* __restrict__ gx,
                                                            act_t* __restrict__ gx16) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float mean = stats[2 * row], rstd = stats[2 * row + 1];
  const XT* xr = x + (size_t)row * x_stride;
  const float4* pr = pos ? reinterpret_cast<const float4*>(pos + (size_t)(row % T) * W) : nullptr;
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  float4* gxr = gx ? reinterpret_cast<float4*>(gx + (size_t)row * x_stride) : nullptr;
  float4 g[NV], xh[NV], prev[NV];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c4 = lane + 32 * i;
    float4 t = ld_x4(xr, c4);
    if (pr) {
      float4 q = pr[c4];
      t.x += q.x;
      t.y += q.y;
      t.z += q.z;
      t.w += q.w;
    }
    if (accumulate) prev[i] = gxr ? gxr[c4] : ld_half4(gx16 + (size_t)row * x_stride + 4 * c4);
    float4 d = ld_half4(dy + (size_t)row * W + 4 * c4), gm = g4[c4];
    xh[i] = make_float4((t.x - mean) * rstd, (t.y - mean) * rstd, (t.z - mean) * rstd, (t.w - mean) * rstd);
    g[i] = make_float4(d.x * gm.x, d.y * gm.y, d.z * gm.z, d.w * gm.w);
    s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
    s2 += (g[i].x * xh[i].x + g[i].y * xh[i].y) + (g[i].z * xh[i].z + g[i].w * xh[i].w);
  }
  s1 = warp_sum(s1) / W;
  s2 = warp_sum(s2) / W;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c4 = lane + 32 * i;
    float4 d;
    d.x = rstd * (g[i].x - s1 - xh[i].x * s2);
    d.y = rstd * (g[i].y - s1 - xh[i].y * s2);
    d.z = rstd * (g[i].z - s1 - xh[i].z * s2);
    d.w = rstd * (g[i].w - s1 - xh[i].w * s2);
    if (accumulate) {
      d.x += prev[i].x;
      d.y += prev[i].y;
      d.z += prev[i].z;
      d.w += prev[i].w;
    }
    if (gxr) gxr[c4] = d;
    if (gx16) st_half4(gx16 + (size_t)row * x_stride + 4 * c4, d.x, d.y, d.z, d.w);
  }
}

// fp16 residual stream, W % 256 == 0: every access is a 16-byte vector of 8 halfs (lane owns NV8 = W / 256 of them per
// tensor) -- half the load / store instructions of the 8-byte form above for the same bytes.
__device__ __forceinline__ void ln_unpack8(const uint4& u, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 ln_pack8(const float (&f)[8]) {
  uint4 u;
  __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
  return u;
}

template <int NV8>
__global__ void __launch_bounds__(256) layernorm_fwd16_kernel(const act_t* __restrict__ x, long long x_stride,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, int rows, int W, float eps,
                                                              act_t* __restrict__ y16, float* __restrict__ stats) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * x_stride);
  uint4 raw[NV8];
#pragma unroll
  for (int i = 0; i < NV8; ++i) raw[i] = xr[lane + 32 * i];
  float v[NV8][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    ln_unpack8(raw[i], v[i]);
#pragma unroll
    for (int j = 0; j < 8; j += 4) s += (v[i][j] + v[i][j + 1]) + (v[i][j + 2] + v[i][j + 3]);
  }
  const float mean = warp_sum(s) / W;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV8; ++i)
#pragma unroll
    for (int j = 0; j < 8; j += 4) {
      const float a = v[i][j] - mean, b = v[i][j + 1] - mean, c = v[i][j + 2] - mean, d = v[i][j + 3] - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  const float rstd = rsqrtf(warp_sum(q) / W + eps);
  if (lane == 0) {
    stats[2 * row] = mean;
    stats[2 * row + 1] = rstd;
  }
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
  uint4* yr = reinterpret_cast<uint4*>(y16 + (size_t)row * W);
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int c8 = lane + 32 * i;
    const float4 ga = g4[2 * c8], gb = g4[2 * c8 + 1], ba = b4[2 * c8], bb = b4[2 * c8 + 1];
    const float g[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
    const float b[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * g[j] + b[j];
    yr[c8] = ln_pack8(o);
  }
}

template <int NV8>
__global__ void __launch_bounds__(256) layernorm_bwd16_kernel(const act_t* __restrict__ dy, const act_t* __restrict__ x,
                                                              long long x_stride, const float* __restrict__ stats,
                                                              const float* __restrict__ gamma, int rows, int W,
                                                              int accumulate, act_t* __restrict__ gx16) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float mean = stats[2 * row], rstd = stats[2 * row + 1];
  const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * x_stride);
  const uint4* dr = reinterpret_cast<const uint4*>(dy + (size_t)row * W);
  uint4* gr = reinterpret_cast<uint4*>(gx16 + (size_t)row * x_stride);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  uint4 rx[NV8], rd[NV8], rp[NV8];
#pragma unroll
  for (int i = 0; i < NV8; ++i) {  // every load of the row in flight before the first use
    rx[i] = xr[lane + 32 * i];
    rd[i] = dr[lane + 32 * i];
    if (accumulate) rp[i] = gr[lane + 32 * i];
  }
  float g[NV8][8], xh[NV8][8];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int c8 = lane + 32 * i;
    const float4 ga = g4[2 * c8], gb = g4[2 * c8 + 1];
    const float gm[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
    float xv[8], dv[8];
    ln_unpack8(rx[i], xv);
    ln_unpack8(rd[i], dv);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      xh[i][j] = (xv[j] - mean) * rstd;
      g[i][j] = dv[j] * gm[j];
    }
#pragma unroll
    for (int j = 0; j < 8; j += 4) {
      s1 += (g[i][j] + g[i][j + 1]) + (g[i][j + 2] + g[i][j + 3]);
      s2 += (g[i][j] * xh[i][j] + g[i][j + 1] * xh[i][j + 1]) + (g[i][j + 2] * xh[i][j + 2] + g[i][j + 3] * xh[i][j + 3]);
    }
  }
  s1 = warp_sum(s1) / W;
  s2 = warp_sum(s2) / W;
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    float d[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] = rstd * (g[i][j] - s1 - xh[i][j] * s2);
    if (accumulate) {
      float pv[8];
      ln_unpack8(rp[i], pv);
#pragma unroll
      for (int j = 0; j < 8; ++j) d[j] += pv[j];
    }
    gr[lane + 32 * i] = ln_pack8(d);
  }
}

// one warp per row; lane owns NV 16-byte vectors (8 halfs) of the row: ld % 8 == 0, ld <= 256 * NV
template <int NV>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(act_t* __restrict__ s, long long rows, int cols, int ld) {
  pdl_prologue();
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  act_t* r = s + row * ld;
  const int nvec = ld / 8;
  float v[NV][8];
  float m = -FLT_MAX;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + 32 * i;
    if (vi < nvec) {
      uint4 u = *reinterpret_cast<const uint4*>(r + vi * 8);
      const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 f = __half22float2(h[j]);
        v[i][2 * j] = f.x;
        v[i][2 * j + 1] = f.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (vi >= nvec || vi * 8 + j >= cols) v[i][j] = -FLT_MAX;
      m = fmaxf(m, v[i][j]);
    }
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = (lane + 32 * i) * 8 + j;
      v[i][j] = (c < cols) ? __expf(v[i][j] - m) : 0.f;
      sum += v[i][j];
    }
  const float inv = 1.f / warp_sum(sum);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + 32 * i;
    if (vi < nvec) {
      uint4 u;
      __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) h[j] = __floats2half2_rn(v[i][2 * j] * inv, v[i][2 * j + 1] * inv);
      *reinterpret_cast<uint4*>(r + vi * 8) = u;
    }
  }
}

template <int NV>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const act_t* __restrict__ p, act_t* __restrict__ dp,
                                                          long long rows, int cols, int ld) {
  pdl_prologue();
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const act_t* pr = p + row * ld;
  act_t* dr = dp + row * ld;
  const int nvec = ld / 8;
  float pv[NV][8], dv[NV][8];
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + 32 * i;
    if (vi < nvec) {
      uint4 a = *reinterpret_cast<const uint4*>(pr + vi * 8), b = *reinterpret_cast<const uint4*>(dr + vi * 8);
      const __half2* ha = reinterpret_cast<const __half2*>(&a);
      const __half2* hb = reinterpret_cast<const __half2*>(&b);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 fa = __half22float2(ha[j]), fb = __half22float2(hb[j]);
        pv[i][2 * j] = fa.x;
        pv[i][2 * j + 1] = fa.y;
        dv[i][2 * j] = fb.x;
        dv[i][2 * j + 1] = fb.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (vi >= nvec || vi * 8 + j >= cols) {
        pv[i][j] = 0.f;
        dv[i][j] = 0.f;
      }
      dot += pv[i][j] * dv[i][j];
    }
  }
  dot = warp_sum(dot);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + 32 * i;
    if (vi < nvec) {
      uint4 u;
      __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        h[j] = __floats2half2_rn(pv[i][2 * j] * (dv[i][2 * j] - dot), pv[i][2 * j + 1] * (dv[i][2 * j + 1] - dot));
      *reinterpret_cast<uint4*>(dr + vi * 8) = u;
    }
  }
}

// one block (128 threads) per cutout row.  Accumulates losses with atomics (n prompts).
__global__ void __launch_bounds__(128) prompt_loss_kernel(const float* __restrict__ e, int D,
                                                          const float* __restrict__ prompts,
                                                          const float* __restrict__ weights,
                                                          const float* __restrict__ stops,
                                                          const int* __restrict__ slots,
                                                          const float* __restrict__ inv_rows, int n, float inv_count,
                                                          float grad_scale, float* __restrict__ e_unit,
                                                          float* __restrict__ losses, float* __restrict__ de,
                                                          act_t* __restrict__ de16) {
  pdl_prologue();
  extern __shared__ float sh[];  // en [D], gen [D]
  float* en = sh;
  float* gen = sh + D;
  __shared__ float red[4];
  __shared__ float s_val;
  const int b = blockIdx.x;
  auto block_sum = [&](float v) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) s_val = red[0] + red[1] + red[2] + red[3];
    __syncthreads();
    return s_val;
  };
  float ss = 0.f;
  for (int d = threadIdx.x; d < D; d += 128) {
    float t = e[(size_t)b * D + d];
    ss += t * t;
  }
  const float nrm = fmaxf(sqrtf(block_sum(ss)), 1e-12f);  // img_embeddings / norm (slip.py:66), F.normalize eps
  for (int d = threadIdx.x; d < D; d += 128) {
    float t = e[(size_t)b * D + d] / nrm;
    en[d] = t;
    gen[d] = 0.f;
    if (e_unit) e_unit[(size_t)b * D + d] = t;
  }
  __syncthreads();
  for (int j = 0; j < n; ++j) {
    const float* pj = prompts + (size_t)j * D;
    float rr = 0.f;
    for (int d = threadIdx.x; d < D; d += 128) {
      float t = en[d] - pj[d];
      rr += t * t;
    }
    const float r = sqrtf(block_sum(rr));
    const float w = weights[j], stop = stops[j];
    const float sgn = (w > 0.f) ? 1.f : ((w < 0.f) ? -1.f : 0.f);
    const float a = asinf(fminf(r * 0.5f, 1.f));
    const float dist = 2.f * a * a * sgn;                // pixray.py:278-279
    // row j of a Prompt whose embed has 1/inv_rows[j] rows (image prompts: [cutn, D], pixray.py:1327-1333); the mean
    // of Prompt.forward runs over [cutn, rows]
    const float inv_n = inv_count * (inv_rows ? inv_rows[j] : 1.f);
    if (threadIdx.x == 0) atomicAdd(&losses[slots ? slots[j] : j], fabsf(w) * dist * inv_n);
    // replace_grad(dists, maximum(dists, stop)): gradient only where dists > stop (pixray.py:280)
    if (dist > stop && r > 0.f) {
      // d dist / d r = sgn * 2 asin(r/2) / sqrt(1 - r^2/4)
      const float ddr = sgn * 2.f * a / sqrtf(fmaxf(1.f - 0.25f * r * r, 1e-12f));
      const float coef = fabsf(w) * inv_n * grad_scale * ddr / r;
      for (int d = threadIdx.x; d < D; d += 128) gen[d] += coef * (en[d] - pj[d]);
    }
    __syncthreads();
  }
  // back through the normalisation: de = (gen - en * <gen, en>) / |e|
  float dot = 0.f;
  for (int d = threadIdx.x; d < D; d += 128) dot += gen[d] * en[d];
  dot = block_sum(dot);
  for (int d = threadIdx.x; d < D; d += 128) {
    float v = (gen[d] - en[d] * dot) / nrm;
    de[(size_t)b * D + d] = v;
    if (de16) de16[(size_t)b * D + d] = __float2half_rn(v);
  }
}

// clip_z after the optimiser step: per-channel [zmin, zmax] (vqgan.py:202-204) or [0, 1] (fast_pixeldrawer.py:98-100)
__device__ __forceinline__ float clip_z_one(float zi, int i, int per_channel, const float* __restrict__ zmin,
                                            const float* __restrict__ zmax, int clip01) {
  if (zmin) {
    const int c = i / per_channel;
    zi = fminf(fmaxf(zi, zmin[c]), zmax[c]);
  } else if (clip01) {
    zi = fminf(fmaxf(zi, 0.f), 1.f);
  }
  return zi;
}

// Adam's moments: m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2, rounded as fma(b1, m, (1 - b1) g) and
// fma(b2, v, ((1 - b2) g) g)
__device__ __forceinline__ float adam_m(float m, float g, float b1) { return __fmaf_rn(b1, m, __fmul_rn(1.f - b1, g)); }
__device__ __forceinline__ float adam_v(float v, float g, float b2) {
  return __fmaf_rn(b2, v, __fmul_rn(__fmul_rn(1.f - b2, g), g));
}

// One optimiser step on element i (see kernels.cuh "optimiser").  Returns the new z (before clip_z) and writes the
// updated state, or zeroes it when `fresh` (the managed kernel's rebuild: the NEXT step starts from a new optimiser).
template <int K>
__device__ __forceinline__ float opt_update(float zi, float gi, const OptState& s, int i, float b1, float b2, float eps,
                                            const OptCoef& c, bool fresh) {
  if constexpr (K == OPT_ADAM || K == OPT_ADAMW) {
    if constexpr (K == OPT_ADAMW) zi = zi * c.decay;  // torch.optim.AdamW: decoupled decay BEFORE the Adam step
    // torch.optim.Adam: step_size = lr / (1 - b1^t); denom = sqrt(v) / sqrt(1 - b2^t) + eps.  The roundings are pinned
    // so that every instantiation keeps the contraction the Adam-only kernels had (same bits as before).
    const float mi = adam_m(s.s0[i], gi, b1);
    const float vi = adam_v(s.s1[i], gi, b2);
    s.s0[i] = fresh ? 0.f : mi;
    s.s1[i] = fresh ? 0.f : vi;
    const float denom = __fmaf_rn(sqrtf(vi), c.inv_sqrt_bc2, eps);
    return zi - __fmul_rn(c.step_size, mi) / denom;
  } else if constexpr (K == OPT_ADAGRAD) {
    // torch.optim.Adagrad (lr_decay 0, initial accumulator 0): sum += g^2; z -= lr * g / (sqrt(sum) + 1e-10)
    const float si = s.s1[i] + gi * gi;
    s.s1[i] = fresh ? 0.f : si;
    return zi - c.step_size * (gi / (sqrtf(si) + 1e-10f));
  } else if constexpr (K == OPT_ADAMAX) {
    // torch.optim.Adamax: m.lerp_(g, 1 - b1); u = max(b2 u, |g| + eps); z -= lr / (1 - b1^t) * m / u
    const float m0 = s.s0[i];
    const float mi = m0 + (1.f - b1) * (gi - m0);
    const float ui = fmaxf(b2 * s.s1[i], fabsf(gi) + eps);
    s.s0[i] = fresh ? 0.f : mi;
    s.s1[i] = fresh ? 0.f : ui;
    return zi - c.step_size * (mi / ui);
  } else {
    static_assert(K == OPT_DIFFGRAD, "unknown optimiser kind");
    // torch_optimizer.DiffGrad 0.1.0: m, v as Adam; denom = sqrt(v) + eps (eps NOT bias-corrected);
    // dfc = 1 / (1 + exp(-|p - g|)); p = g; z -= lr sqrt(1 - b2^t) / (1 - b1^t) * (m dfc) / denom
    const float mi = adam_m(s.s0[i], gi, b1);
    const float vi = adam_v(s.s1[i], gi, b2);
    const float dfc = 1.f / (1.f + expf(-fabsf(s.s2[i] - gi)));
    s.s0[i] = fresh ? 0.f : mi;
    s.s1[i] = fresh ? 0.f : vi;
    s.s2[i] = fresh ? 0.f : gi;
    const float denom = sqrtf(vi) + eps;
    return zi - c.step_size * ((mi * dfc) / denom);
  }
}

template <int K>
__global__ void opt_clip_kernel(float* __restrict__ z, OptState s, const float* __restrict__ g, float inv_scale, int n,
                                int per_channel, const float* __restrict__ zmin, const float* __restrict__ zmax,
                                int clip01, float b1, float b2, float eps, OptCoef c) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * inv_scale;
  const float zi = opt_update<K>(z[i], gi, s, i, b1, b2, eps, c, false);
  z[i] = clip_z_one(zi, i, per_channel, zmin, zmax, clip01);
}

// see kernels.cuh "device-side checkdrop + optimiser step"
template <int K>
__global__ void opt_clip_managed_kernel(float* __restrict__ z, OptState s, const float* __restrict__ g,
                                        float* __restrict__ best_z, float inv_scale, int n, int per_channel,
                                        const float* __restrict__ zmin, const float* __restrict__ zmax, int clip01,
                                        float b1, float b2, float eps, const float* __restrict__ losses, int n_losses,
                                        int iter, DropConfig cfg, const DropState* __restrict__ cur,
                                        DropState* __restrict__ next, DropStatus* status) {
  pdl_prologue();
  const DropState ds = *cur;
  const bool writer = blockIdx.x == 0 && threadIdx.x == 0;
  float loss_sum = 0.f;
  for (int k = 0; k < n_losses; ++k) loss_sum += losses[k];  // sum(lossAll): left to right in fp32 like Python's sum()
  DropState nx = ds;
  bool rebuild = false, new_best = false;
  if (!ds.stopped) {
    bool scheduled = false;
    for (int k = 0; k < cfg.n_sched; ++k) scheduled |= (cfg.sched[k] == iter);
    if (scheduled) {
      rebuild = true;  // "Dropping learning rate" (pixray.py:1468-1470): checkdrop is not consulted on these iterations
    } else {
      bool drop = false;
      if (loss_sum < ds.best_loss) {
        new_best = true;
        nx.best_loss = loss_sum;
        nx.best_iter = iter;
      } else if (iter - ds.best_iter >= cfg.iter_drop_delay) {
        drop = true;
      }
      if (cfg.auto_stop) rebuild = drop;
    }
    const int t = ds.adam_t + 1;
    nx.adam_t = t;
    const OptCoef c = opt_coef(K, ds.lr, b1, b2, t);
    if (rebuild) {
      nx.num_loss_drop = ds.num_loss_drop + 1;
      if (nx.num_loss_drop > cfg.max_loss_drops) {
        nx.stopped = 1;  // train() returns False (pixray.py:1505-1506); this iteration's step still happened
      } else {
        nx.best_iter = iter;
        nx.best_loss = 1e20f;
        nx.adam_t = 0;
        nx.lr = (float)((double)cfg.base_lr / pow(10.0, (double)nx.num_loss_drop));  // learning_rate / 10^drops (pixray.py:522-539)
      }
    }
    const bool fresh = rebuild && !nx.stopped;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
      const float z0 = z[i];
      if (new_best && best_z) best_z[i] = z0;  // best_z = drawer.get_z_copy() (pixray.py:1104): z BEFORE this step
      const float gi = g[i] * inv_scale;
      const float zi = opt_update<K>(z0, gi, s, i, b1, b2, eps, c, fresh);
      z[i] = clip_z_one(zi, i, per_channel, zmin, zmax, clip01);
    }
  }
  if (writer) {
    *next = nx;
    if (status) {
      status->seq_begin = iter + 1;
      __threadfence_system();
      status->iter = iter;
      status->loss_sum = loss_sum;
      status->best_loss = nx.best_loss;
      status->best_iter = nx.best_iter;
      status->num_loss_drop = nx.num_loss_drop;
      status->stopped = nx.stopped;
      status->rebuilt = rebuild ? 1 : 0;
      status->lr = nx.lr;
      status->n_losses = n_losses;
      for (int k = 0; k < n_losses && k < 64; ++k) status->losses[k] = losses[k];
      __threadfence_system();
      status->seq_end = iter + 1;
    }
  }
}

__global__ void accumulate_kernel(const float* __restrict__ g, float* __restrict__ acc, long long n, int accumulate) {
  pdl_prologue();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc[i] = accumulate ? acc[i] + g[i] : g[i];
}

__global__ void fill_kernel(float* p, float v, long long n) {
  pdl_prologue();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] = v;
}
__global__ void cast_kernel(const float* x, act_t* y, long long n, float scale) {
  pdl_prologue();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = __float2half_rn(x[i] * scale);
}

}  // namespace

// PXR_LN16_WIDE=0 keeps the 8-byte-vector LayerNorm kernels on the fp16 stream (A/B switch)
static bool ln16_wide_ok() {
  static const bool on = [] {
    const char* e = getenv("PXR_LN16_WIDE");
    return !(e && atoi(e) == 0);
  }();
  return on;
}

#define LN_DISPATCH(KERNEL, XT, ...)                                                   \
  switch (W / 128) {                                                              \
    case 1: launch_pdl(KERNEL<1, XT>, dim3((rows + 7) / 8), dim3(256), 0, st, __VA_ARGS__); break;        \
    case 2: launch_pdl(KERNEL<2, XT>, dim3((rows + 7) / 8), dim3(256), 0, st, __VA_ARGS__); break;        \
    case 4: launch_pdl(KERNEL<4, XT>, dim3((rows + 7) / 8), dim3(256), 0, st, __VA_ARGS__); break;        \
    case 6: launch_pdl(KERNEL<6, XT>, dim3((rows + 7) / 8), dim3(256), 0, st, __VA_ARGS__); break;        \
    case 8: launch_pdl(KERNEL<8, XT>, dim3((rows + 7) / 8), dim3(256), 0, st, __VA_ARGS__); break;        \
    default: break;                                                               \
  }

void layernorm_forward(const float* x, long long x_stride, const float* pos, int T, const float* gamma,
                       const float* beta, int rows, int W, float eps, act_t* y16, float* y32, float* stats,
                       cudaStream_t st) {
  LN_DISPATCH(layernorm_fwd_kernel, float, x, x_stride, pos, T, gamma, beta, rows, W, eps, y16, y32, stats)
}
void layernorm_forward(const act_t* x, long long x_stride, const float* pos, int T, const float* gamma,
                       const float* beta, int rows, int W, float eps, act_t* y16, float* y32, float* stats,
                       cudaStream_t st) {
  if (ln16_wide_ok() && !pos && !y32 && y16 && W % 256 == 0 && x_stride % 8 == 0) {
    const dim3 grid((rows + 7) / 8), block(256);
    switch (W / 256) {
      case 1: launch_pdl(layernorm_fwd16_kernel<1>, grid, block, 0, st, x, x_stride, gamma, beta, rows, W, eps, y16, stats); return;
      case 2: launch_pdl(layernorm_fwd16_kernel<2>, grid, block, 0, st, x, x_stride, gamma, beta, rows, W, eps, y16, stats); return;
      case 3: launch_pdl(layernorm_fwd16_kernel<3>, grid, block, 0, st, x, x_stride, gamma, beta, rows, W, eps, y16, stats); return;
      case 4: launch_pdl(layernorm_fwd16_kernel<4>, grid, block, 0, st, x, x_stride, gamma, beta, rows, W, eps, y16, stats); return;
      default: break;
    }
  }
  LN_DISPATCH(layernorm_fwd_kernel, act_t, x, x_stride, pos, T, gamma, beta, rows, W, eps, y16, y32, stats)
}
void layernorm_backward(const act_t* dy, const float* x, long long x_stride, const float* pos, int T,
                        const float* stats, const float* gamma, int rows, int W, int accumulate, float* gx,
                        act_t* gx16, cudaStream_t st) {
  LN_DISPATCH(layernorm_bwd_kernel, float, dy, x, x_stride, pos, T, stats, gamma, rows, W, accumulate, gx, gx16)
}
void layernorm_backward(const act_t* dy, const act_t* x, long long x_stride, const float* pos, int T,
                        const float* stats, const float* gamma, int rows, int W, int accumulate, float* gx,
                        act_t* gx16, cudaStream_t st) {
  if (ln16_wide_ok() && !pos && !gx && gx16 && W % 256 == 0 && x_stride % 8 == 0) {
    const dim3 grid((rows + 7) / 8), block(256);
    switch (W / 256) {
      case 1: launch_pdl(layernorm_bwd16_kernel<1>, grid, block, 0, st, dy, x, x_stride, stats, gamma, rows, W, accumulate, gx16); return;
      case 2: launch_pdl(layernorm_bwd16_kernel<2>, grid, block, 0, st, dy, x, x_stride, stats, gamma, rows, W, accumulate, gx16); return;
      case 3: launch_pdl(layernorm_bwd16_kernel<3>, grid, block, 0, st, dy, x, x_stride, stats, gamma, rows, W, accumulate, gx16); return;
      case 4: launch_pdl(layernorm_bwd16_kernel<4>, grid, block, 0, st, dy, x, x_stride, stats, gamma, rows, W, accumulate, gx16); return;
      default: break;
    }
  }
  LN_DISPATCH(layernorm_bwd_kernel, act_t, dy, x, x_stride, pos, T, stats, gamma, rows, W, accumulate, gx, gx16)
}
void softmax_forward(act_t* s, int rows, int cols, int ld, cudaStream_t st) {
  const int nv = (ld / 8 + 31) / 32;
  const int grid = (rows + 7) / 8;
  if (nv <= 1) launch_pdl(softmax_fwd_kernel<1>, dim3(grid), dim3(256), 0, st, s, rows, cols, ld);
  else if (nv == 2) launch_pdl(softmax_fwd_kernel<2>, dim3(grid), dim3(256), 0, st, s, rows, cols, ld);
  else launch_pdl(softmax_fwd_kernel<4>, dim3(grid), dim3(256), 0, st, s, rows, cols, ld);
}
void softmax_backward(const act_t* p, act_t* dp_to_ds, int rows, int cols, int ld, cudaStream_t st) {
  const int nv = (ld / 8 + 31) / 32;
  const int grid = (rows + 7) / 8;
  if (nv <= 1) launch_pdl(softmax_bwd_kernel<1>, dim3(grid), dim3(256), 0, st, p, dp_to_ds, rows, cols, ld);
  else if (nv == 2) launch_pdl(softmax_bwd_kernel<2>, dim3(grid), dim3(256), 0, st, p, dp_to_ds, rows, cols, ld);
  else launch_pdl(softmax_bwd_kernel<4>, dim3(grid), dim3(256), 0, st, p, dp_to_ds, rows, cols, ld);
}
void prompt_loss(const float* e, int B, int D, const float* prompts, const float* weights, const float* stops,
                 const int* slots, const float* inv_rows, int n, int cutn_global, float grad_scale, float* e_unit,
                 float* losses, float* de, act_t* de16, cudaStream_t st) {
  // Prompt.forward means over [cutn, n_embed] per prompt (pixray.py:280)
  launch_pdl(prompt_loss_kernel, dim3(B), dim3(128), 2 * D * sizeof(float), st, e, D, prompts, weights, stops, slots, inv_rows, n,
                                                           1.f / cutn_global, grad_scale, e_unit, losses, de, de16);
}

#define OPT_DISPATCH(KERNEL, GRID, ...)                                                                 \
  switch (kind) {                                                                                       \
    case OPT_ADAM: launch_pdl(KERNEL<OPT_ADAM>, GRID, dim3(256), 0, st, __VA_ARGS__); break;            \
    case OPT_ADAMW: launch_pdl(KERNEL<OPT_ADAMW>, GRID, dim3(256), 0, st, __VA_ARGS__); break;          \
    case OPT_ADAGRAD: launch_pdl(KERNEL<OPT_ADAGRAD>, GRID, dim3(256), 0, st, __VA_ARGS__); break;      \
    case OPT_ADAMAX: launch_pdl(KERNEL<OPT_ADAMAX>, GRID, dim3(256), 0, st, __VA_ARGS__); break;        \
    case OPT_DIFFGRAD: launch_pdl(KERNEL<OPT_DIFFGRAD>, GRID, dim3(256), 0, st, __VA_ARGS__); break;    \
    default: throw std::runtime_error("unknown optimiser kind");                                        \
  }

void opt_clip_step(int kind, float* z, OptState s, const float* g, float inv_scale, int n, int per_channel,
                   const float* zmin, const float* zmax, int clip01, float lr, float b1, float b2, float eps, int t,
                   cudaStream_t st) {
  const OptCoef c = opt_coef(kind, lr, b1, b2, t);
  OPT_DISPATCH(opt_clip_kernel, dim3((n + 255) / 256), z, s, g, inv_scale, n, per_channel, zmin, zmax, clip01, b1, b2,
               eps, c)
}

void opt_clip_managed(int kind, float* z, OptState s, const float* g, float* best_z, float inv_scale, int n,
                      int per_channel, const float* zmin, const float* zmax, int clip01, float b1, float b2, float eps,
                      const float* losses, int n_losses, int iter, const DropConfig& cfg, const DropState* cur,
                      DropState* next, DropStatus* status_mapped, cudaStream_t st) {
  int grid = (n + 255) / 256;
  if (grid > 148 * 4) grid = 148 * 4;
  OPT_DISPATCH(opt_clip_managed_kernel, dim3(grid), z, s, g, best_z, inv_scale, n, per_channel, zmin, zmax, clip01, b1,
               b2, eps, losses, n_losses, iter, cfg, cur, next, status_mapped)
}

void accumulate_f32(const float* g, float* acc, long long n, int accumulate, cudaStream_t st) {
  long long gr = (n + 255) / 256;
  if (gr > 148 * 8) gr = 148 * 8;
  launch_pdl(accumulate_kernel, dim3((int)gr), dim3(256), 0, st, g, acc, n, accumulate);
}

void fill_f32(float* p, float v, long long n, cudaStream_t st) {
  long long g = (n + 255) / 256;
  if (g > 148 * 8) g = 148 * 8;
  launch_pdl(fill_kernel, dim3((int)g), dim3(256), 0, st, p, v, n);
}
void cast_f32_to_f16(const float* x, act_t* y, long long n, float scale, cudaStream_t st) {
  long long g = (n + 255) / 256;
  if (g > 148 * 8) g = 148 * 8;
  launch_pdl(cast_kernel, dim3((int)g), dim3(256), 0, st, x, y, n, scale);
}

}  // namespace pxr
