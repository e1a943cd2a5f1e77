// FP32 correctness mode of the DPT path (SURVEY.md 8c: "fp32: kernel(fp32 mode) vs oracle(fp32) rel-L2 <= 1e-5 at
// every tap").  The reference is fp32-only (omnidata_tools/torch/requirements.txt:4, no autocast anywhere); this
// file evaluates the same contractions on the FP32 FMA pipe so that the production bf16 tensor-core path has an
// in-repo fp32 twin with the same data flow, layouts, fusions and launch order:
//   conv_f32_kernel       implicit-GEMM convolution / linear layer over the same odb_conv_gemm_desc (strided
//                         channels-last views, taps, bias / act / residual / relu copy), 64 x 64 output tile per CTA,
//                         K blocks of 32; every K block is accumulated in fp32 and the block sums are combined in
//                         fp64, so the result is closer to exact arithmetic than a sequential fp32 dot product
//   attention_f32_kernel  softmax(q k^T * scale) v with fp64 dot products (timm Attention.forward)
//   head_tail_f32_kernel  the 1x1 conv (+ReLU) that ends the DPT head, NHWC -> NCHW (dpt_depth.py:95-97)
// Compiled WITHOUT --use_fast_math (exact division, erff, expf).  Speed is not the point of this mode.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "host_util.h"
#include "../../include/omnidata_b200.h"

namespace odb {

constexpr int kF32BM = 64, kF32BN = 64, kF32BK = 32, kF32Pad = 4;

struct ConvF32Params {
  const float* view[ODB_MAX_VIEWS];
  int vw[ODB_MAX_VIEWS], vh[ODB_MAX_VIEWS];
  long long vsx[ODB_MAX_VIEWS], vsy[ODB_MAX_VIEWS], vsb[ODB_MAX_VIEWS];
  int C, num_taps;
  int8_t tap_view[ODB_MAX_TAPS], tap_dx[ODB_MAX_TAPS], tap_dy[ODB_MAX_TAPS];
  const float* weight;   // [N][num_taps * C]
  int N;
  float* out;  long long osx, osy, osb;
  float* out2; long long o2sx, o2sy, o2sb;
  const float* bias; long long bias_sb;
  const float* res;  long long rsx, rsy, rsb;
  int act;
  int ow, oh, ob;
};

__global__ void __launch_bounds__(256) conv_f32_kernel(const __grid_constant__ ConvF32Params p) {
  __shared__ float As[kF32BK][kF32BM + kF32Pad];   // [k][pixel]
  __shared__ float Bs[kF32BK][kF32BN + kF32Pad];   // [k][out channel]
  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;              // 16 x 16 threads, 4 x 4 outputs each
  const long long M = (long long)p.ob * p.oh * p.ow;
  const long long m0 = (long long)blockIdx.x * kF32BM;
  const int n0 = blockIdx.y * kF32BN;
  const int K = p.num_taps * p.C;

  // the two (pixel, 4-channel group) items this thread stages per K block
  int lp[2], lc[2], lb[2], ly[2], lx[2];
  bool lvalid[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int idx = t * 2 + i;
    lp[i] = idx >> 3;
    lc[i] = (idx & 7) * 4;
    const long long m = m0 + lp[i];
    lvalid[i] = m < M;
    const long long mm = lvalid[i] ? m : 0;
    lx[i] = (int)(mm % p.ow);
    ly[i] = (int)((mm / p.ow) % p.oh);
    lb[i] = (int)(mm / ((long long)p.ow * p.oh));
  }

  double accd[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) accd[i][j] = 0.0;

  for (int tap = 0; tap < p.num_taps; ++tap) {
    const int v = p.tap_view[tap];
    const float* vbase = p.view[v];
    for (int c0 = 0; c0 < p.C; c0 += kF32BK) {
      // ---- stage A (gathered input pixels; out of range = zero padding) and B (weights), transposed to [k][.]
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        const int yy = ly[i] + p.tap_dy[tap], xx = lx[i] + p.tap_dx[tap];
        if (lvalid[i] && yy >= 0 && yy < p.vh[v] && xx >= 0 && xx < p.vw[v] && c0 + lc[i] < p.C)
          a = *reinterpret_cast<const float4*>(vbase + lb[i] * p.vsb[v] + yy * p.vsy[v] + xx * p.vsx[v] + c0 + lc[i]);
        As[lc[i] + 0][lp[i]] = a.x; As[lc[i] + 1][lp[i]] = a.y; As[lc[i] + 2][lp[i]] = a.z; As[lc[i] + 3][lp[i]] = a.w;
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        const int n = n0 + lp[i];
        if (n < p.N && c0 + lc[i] < p.C)
          b = *reinterpret_cast<const float4*>(p.weight + (long long)n * K + (long long)tap * p.C + c0 + lc[i]);
        Bs[lc[i] + 0][lp[i]] = b.x; Bs[lc[i] + 1][lp[i]] = b.y; Bs[lc[i] + 2][lp[i]] = b.z; Bs[lc[i] + 3][lp[i]] = b.w;
      }
      __syncthreads();
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll
      for (int k = 0; k < kF32BK; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) accd[i][j] += (double)acc[i][j];
      __syncthreads();
    }
  }

  // ---- epilogue: residual + act(acc + bias); optional relu copy
  const int n = n0 + tx * 4;
  if (n >= p.N) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
    const int x = (int)(m % p.ow), y = (int)((m / p.ow) % p.oh), b = (int)(m / ((long long)p.ow * p.oh));
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float bias = p.bias ? p.bias[(long long)b * p.bias_sb + n + j] : 0.f;
      float r = (float)(accd[i][j] + (double)bias);
      if (p.act == ODB_ACT_RELU) r = fmaxf(r, 0.f);
      else if (p.act == ODB_ACT_GELU) r = 0.5f * r * (1.0f + erff(r * 0.70710678118654752440f));
      v[j] = r;
    }
    if (p.res) {
      const float4 r4 = *reinterpret_cast<const float4*>(p.res + b * p.rsb + y * p.rsy + x * p.rsx + n);
      v[0] += r4.x; v[1] += r4.y; v[2] += r4.z; v[3] += r4.w;
    }
    *reinterpret_cast<float4*>(p.out + b * p.osb + y * p.osy + x * p.osx + n) = make_float4(v[0], v[1], v[2], v[3]);
    if (p.out2)
      *reinterpret_cast<float4*>(p.out2 + b * p.o2sb + y * p.o2sy + x * p.o2sx + n) =
          make_float4(fmaxf(v[0], 0.f), fmaxf(v[1], 0.f), fmaxf(v[2], 0.f), fmaxf(v[3], 0.f));
  }
}

// ------------------------------------------------------------------------------------------ attention
constexpr int kAttQ = 16;          // query rows per CTA
constexpr int kAttMaxTok = 640;

__global__ void __launch_bounds__(256) attention_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                            int tokens, int heads, float scale) {
  __shared__ float q_s[kAttQ][64];
  __shared__ float s_s[kAttQ][kAttMaxTok];
  __shared__ float l_s[kAttQ];
  const int t = threadIdx.x;
  const int q0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const long long row_stride = 3LL * heads * 64;
  const float* base = qkv + (long long)b * tokens * row_stride + h * 64;
  for (int i = t; i < kAttQ * 64; i += 256) {
    const int r = i >> 6, d = i & 63;
    q_s[r][d] = (q0 + r < tokens) ? base[(long long)(q0 + r) * row_stride + d] : 0.f;
  }
  __syncthreads();
  // S = (q k^T) * scale
  for (int idx = t; idx < kAttQ * tokens; idx += 256) {
    const int r = idx & (kAttQ - 1), j = idx / kAttQ;
    const float* kr = base + (long long)j * row_stride + heads * 64;
    double acc = 0.0;
#pragma unroll 16
    for (int d = 0; d < 64; ++d) acc += (double)q_s[r][d] * (double)kr[d];
    s_s[r][j] = (float)acc * scale;
  }
  __syncthreads();
  // softmax rows: warp w owns rows w and w + 8
  const int warp = t >> 5, lane = t & 31;
  for (int r = warp; r < kAttQ; r += 8) {
    float mx = -INFINITY;
    for (int j = lane; j < tokens; j += 32) mx = fmaxf(mx, s_s[r][j]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    double sum = 0.0;
    for (int j = lane; j < tokens; j += 32) {
      const float e = expf(s_s[r][j] - mx);
      s_s[r][j] = e;
      sum += (double)e;
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) l_s[r] = (float)sum;
  }
  __syncthreads();
  // O = P V / l
  const int r = t >> 4, d4 = (t & 15) * 4;
  if (q0 + r < tokens) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    const float* vb = base + 2 * heads * 64 + d4;
    for (int j = 0; j < tokens; ++j) {
      const double pj = (double)s_s[r][j];
      const float4 v = *reinterpret_cast<const float4*>(vb + (long long)j * row_stride);
      a0 += pj * (double)v.x; a1 += pj * (double)v.y; a2 += pj * (double)v.z; a3 += pj * (double)v.w;
    }
    const double inv = 1.0 / (double)l_s[r];
    float* o = out + ((long long)b * tokens + q0 + r) * (heads * 64) + h * 64 + d4;
    *reinterpret_cast<float4*>(o) = make_float4((float)(a0 * inv), (float)(a1 * inv), (float)(a2 * inv), (float)(a3 * inv));
  }
}

// Above kAttMaxTok tokens a score row no longer fits in shared memory.  This kernel keeps none: it makes three
// passes over the keys, kAttKC at a time (K chunk staged in shared memory): the row maximum, the fp64 sum of
// expf(s - max), then O = P V / l in fp64 with s and the exponential recomputed.  The definitions (fp64 dot
// products, s = (float)dot * scale, p = expf(s - max), l rounded to fp32) are those of attention_f32_kernel.
constexpr int kAttKC = 64;

__global__ void __launch_bounds__(256) attention_f32_stream_kernel(const float* __restrict__ qkv,
                                                                   float* __restrict__ out, int tokens, int heads,
                                                                   float scale) {
  __shared__ float q_s[kAttQ][65];
  __shared__ float k_s[kAttKC][65];
  __shared__ float s_s[kAttQ][kAttKC];
  __shared__ float m_s[kAttQ];
  __shared__ float l_s[kAttQ];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int q0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const long long row_stride = 3LL * heads * 64;
  const float* base = qkv + (long long)b * tokens * row_stride + h * 64;
  for (int i = t; i < kAttQ * 64; i += 256) {
    const int r = i >> 6, d = i & 63;
    q_s[r][d] = (q0 + r < tokens) ? base[(long long)(q0 + r) * row_stride + d] : 0.f;
  }
  // row reductions: warp w owns rows w and w + 8; PV: thread t owns row t / 16, head dims 4 (t % 16) ..
  float mx_part[2] = {-INFINITY, -INFINITY};
  double l_part[2] = {0.0, 0.0};
  const int r = t >> 4, d4 = (t & 15) * 4;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  for (int pass = 0; pass < 3; ++pass) {
    for (int j0 = 0; j0 < tokens; j0 += kAttKC) {
      const int nk = tokens - j0 < kAttKC ? tokens - j0 : kAttKC;
      __syncthreads();                       // the previous chunk is consumed; q_s, m_s and l_s are visible
      for (int i = t; i < nk * 16; i += 256) {
        const int jj = i >> 4, dk = (i & 15) * 4;
        const float4 v = *reinterpret_cast<const float4*>(base + (long long)(j0 + jj) * row_stride + heads * 64 + dk);
        k_s[jj][dk] = v.x; k_s[jj][dk + 1] = v.y; k_s[jj][dk + 2] = v.z; k_s[jj][dk + 3] = v.w;
      }
      __syncthreads();
      for (int idx = t; idx < kAttQ * nk; idx += 256) {
        const int rr = idx & (kAttQ - 1), jj = idx / kAttQ;
        double acc = 0.0;
#pragma unroll 16
        for (int d = 0; d < 64; ++d) acc += (double)q_s[rr][d] * (double)k_s[jj][d];
        s_s[rr][jj] = (float)acc * scale;
      }
      __syncthreads();
      if (pass == 0) {
#pragma unroll
        for (int k = 0; k < 2; ++k)
          for (int jj = lane; jj < nk; jj += 32) mx_part[k] = fmaxf(mx_part[k], s_s[warp + 8 * k][jj]);
      } else if (pass == 1) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float m = m_s[warp + 8 * k];
          for (int jj = lane; jj < nk; jj += 32) l_part[k] += (double)expf(s_s[warp + 8 * k][jj] - m);
        }
      } else if (q0 + r < tokens) {
        const float m = m_s[r];
        const float* vb = base + 2 * heads * 64 + d4;
        for (int jj = 0; jj < nk; ++jj) {
          const double pj = (double)expf(s_s[r][jj] - m);
          const float4 v = *reinterpret_cast<const float4*>(vb + (long long)(j0 + jj) * row_stride);
          a0 += pj * (double)v.x; a1 += pj * (double)v.y; a2 += pj * (double)v.z; a3 += pj * (double)v.w;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (pass == 0) {
        float mx = mx_part[k];
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) m_s[warp + 8 * k] = mx;
      } else if (pass == 1) {
        double sum = l_part[k];
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) l_s[warp + 8 * k] = (float)sum;
      }
    }
  }
  __syncthreads();
  if (q0 + r < tokens) {
    const double inv = 1.0 / (double)l_s[r];
    float* o = out + ((long long)b * tokens + q0 + r) * (heads * 64) + h * 64 + d4;
    *reinterpret_cast<float4*>(o) = make_float4((float)(a0 * inv), (float)(a1 * inv), (float)(a2 * inv), (float)(a3 * inv));
  }
}

// ------------------------------------------------------------------------------------------ head tail
__global__ void __launch_bounds__(256) head_tail_f32_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ bias, float* __restrict__ out,
                                                            float* __restrict__ pre, long long pixels_per_image,
                                                            int batch, int head_c, int relu) {
  const long long total = pixels_per_image * batch;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float v[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 a = *reinterpret_cast<const float4*>(x + i * 32 + j * 4);
      v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
    }
    const long long b = i / pixels_per_image, pix = i - b * pixels_per_image;
    for (int k = 0; k < head_c; ++k) {
      double acc = (double)bias[k];
#pragma unroll
      for (int j = 0; j < 32; ++j) acc += (double)v[j] * (double)w[k * 32 + j];
      const float o = (float)acc;
      const long long dst = (b * head_c + k) * pixels_per_image + pix;
      if (pre) pre[dst] = o;
      out[dst] = relu ? fmaxf(o, 0.f) : o;
    }
  }
}

static bool view_ok(const odb_view& v) {
  return v.ptr != nullptr && (reinterpret_cast<uintptr_t>(v.ptr) & 15u) == 0 && v.c % 4 == 0 && v.sx % 4 == 0 &&
         v.sy % 4 == 0 && v.sb % 4 == 0;
}
static void fill_strides(const odb_view& v, long long* sx, long long* sy, long long* sb) {
  *sx = v.sx; *sy = v.sy; *sb = v.sb;
  if (v.w == 1 && *sx == 0) *sx = v.c;
  if (v.h == 1 && *sy == 0) *sy = (long long)v.w * *sx;
}

// called by odb_conv_gemm when desc->in_dtype == ODB_DTYPE_F32
int conv_gemm_f32(const odb_conv_gemm_desc* d, cudaStream_t stream) {
  if (d->out_dtype != ODB_DTYPE_F32) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): out_dtype must be fp32");
  if (d->num_views < 1 || d->num_views > ODB_MAX_VIEWS || d->num_taps < 1 || d->num_taps > ODB_MAX_TAPS)
    return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad view/tap count");
  if (d->head_out != nullptr || d->gn_partial != nullptr)
    return fail(ODB_ERR_UNSUPPORTED, "conv_gemm (fp32 mode): head tail / fused GroupNorm statistics are separate kernels");
  ConvF32Params p;
  memset(&p, 0, sizeof(p));
  p.C = d->views[0].c;
  if (p.C % 4 != 0 || d->n % 4 != 0) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): C and n must be multiples of 4");
  for (int v = 0; v < d->num_views; ++v) {
    if (!view_ok(d->views[v]) || d->views[v].c != p.C) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad view");
    p.view[v] = static_cast<const float*>(d->views[v].ptr);
    p.vw[v] = d->views[v].w; p.vh[v] = d->views[v].h;
    fill_strides(d->views[v], &p.vsx[v], &p.vsy[v], &p.vsb[v]);
  }
  p.num_taps = d->num_taps;
  for (int t = 0; t < d->num_taps; ++t) {
    if (d->tap_view[t] < 0 || d->tap_view[t] >= d->num_views) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad tap");
    p.tap_view[t] = d->tap_view[t]; p.tap_dx[t] = d->tap_dx[t]; p.tap_dy[t] = d->tap_dy[t];
  }
  if (d->weight == nullptr || (reinterpret_cast<uintptr_t>(d->weight) & 15u)) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): weight");
  p.weight = static_cast<const float*>(d->weight);
  p.N = d->n;
  if (!view_ok(d->out) || d->out.c != d->n) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad output view");
  p.out = static_cast<float*>(const_cast<void*>(d->out.ptr));
  fill_strides(d->out, &p.osx, &p.osy, &p.osb);
  p.ow = d->out.w; p.oh = d->out.h; p.ob = d->out.b;
  if (p.ow < 1 || p.oh < 1 || p.ob < 1) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): empty output extent");
  if (d->out2.ptr) {
    if (d->out2_act == ODB_ACT_GELU) return fail(ODB_ERR_UNSUPPORTED, "conv_gemm (fp32 mode): the out2 copy is relu only");
    if (!view_ok(d->out2)) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad out2 view");
    p.out2 = static_cast<float*>(const_cast<void*>(d->out2.ptr));
    fill_strides(d->out2, &p.o2sx, &p.o2sy, &p.o2sb);
  }
  p.bias = d->bias; p.bias_sb = d->bias_sb;
  if (d->residual.ptr) {
    if (!view_ok(d->residual)) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): bad residual view");
    p.res = static_cast<const float*>(d->residual.ptr);
    p.rsx = d->residual.sx; p.rsy = d->residual.sy; p.rsb = d->residual.sb;   // sb may be 0 (batch broadcast)
    if (d->residual.w == 1 && p.rsx == 0) p.rsx = d->residual.c;
    if (d->residual.h == 1 && p.rsy == 0) p.rsy = (long long)d->residual.w * p.rsx;
  }
  p.act = d->act;
  const long long M = (long long)p.ob * p.oh * p.ow;
  const long long gx = (M + kF32BM - 1) / kF32BM;
  if (gx > 0x7fffffffLL) return fail(ODB_ERR_INVALID, "conv_gemm (fp32 mode): too many tiles");
  dim3 grid((unsigned)gx, (unsigned)((p.N + kF32BN - 1) / kF32BN));
  conv_f32_kernel<<<grid, 256, 0, stream>>>(p);
  count_launch();
  return check_launch("conv_gemm (fp32 mode)");
}

}  // namespace odb

using namespace odb;

extern "C" int odb_attention_f32(const float* qkv, float* out, int32_t b, int32_t tokens, int32_t heads, float scale,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!qkv || !out || b < 1 || heads < 1 || tokens < 1) return fail(ODB_ERR_INVALID, "attention_f32: bad argument");
  if ((reinterpret_cast<uintptr_t>(qkv) & 15u) || (reinterpret_cast<uintptr_t>(out) & 15u))
    return fail(ODB_ERR_INVALID, "attention_f32: pointers must be 16-byte aligned");
  dim3 grid((tokens + kAttQ - 1) / kAttQ, heads, b);
  if (tokens <= kAttMaxTok)
    attention_f32_kernel<<<grid, 256, 0, stream>>>(qkv, out, tokens, heads, scale);
  else
    attention_f32_stream_kernel<<<grid, 256, 0, stream>>>(qkv, out, tokens, heads, scale);
  count_launch();
  return check_launch("attention_f32");
}

extern "C" int odb_head_tail_f32(const float* x, const float* w, const float* bias, float* out, float* pre, int32_t b,
                                 int32_t h, int32_t wd, int32_t head_c, int32_t relu, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!x || !w || !bias || !out || b < 1 || h < 1 || wd < 1 || head_c < 1)
    return fail(ODB_ERR_INVALID, "head_tail_f32: bad argument");
  const long long ppi = (long long)h * wd;
  long long blocks = (ppi * b + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  head_tail_f32_kernel<<<(unsigned)blocks, 256, 0, stream>>>(x, w, bias, out, pre, ppi, b, head_c, relu);
  count_launch();
  return check_launch("head_tail_f32");
}

// ============================================================================================ backward, fp32 mode
namespace odb {

// ---- weight gradient of a (strided / multi-view) convolution:  out[n][t * C + c] = sum_{b,y,x} dY[b,y,x,n] * X_t[b,y+dy,x+dx,c]
// 64 x 64 tile of (n, c) per CTA and tap; the pixel range is split over gridDim.z, each split writing its own fp32
// partial (ordered reduction afterwards).  K blocks of 32 pixels in fp32, block sums combined in fp64.
struct WgradF32Params {
  const float* view[ODB_MAX_VIEWS];
  int vw[ODB_MAX_VIEWS], vh[ODB_MAX_VIEWS];
  long long vsx[ODB_MAX_VIEWS], vsy[ODB_MAX_VIEWS], vsb[ODB_MAX_VIEWS];
  int C, num_taps;
  int8_t tap_view[ODB_MAX_TAPS], tap_dx[ODB_MAX_TAPS], tap_dy[ODB_MAX_TAPS];
  const float* dy; long long dsx, dsy, dsb;
  int N, ow, oh, ob;
  float* partial;            // [splits][N][taps * C]
  long long pixels_per_split;
};

__global__ void __launch_bounds__(256) wgrad_f32_kernel(const __grid_constant__ WgradF32Params p) {
  __shared__ float As[kF32BK][kF32BM + kF32Pad];   // [pixel][n]
  __shared__ float Bs[kF32BK][kF32BN + kF32Pad];   // [pixel][c]
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int n0 = blockIdx.x * 64;
  const int c_tiles = (p.C + 63) / 64;
  const int tap = blockIdx.y / c_tiles, c0 = (blockIdx.y % c_tiles) * 64;
  const int v = p.tap_view[tap];
  const long long M = (long long)p.ob * p.oh * p.ow;
  const long long m_begin = (long long)blockIdx.z * p.pixels_per_split;
  const long long m_end = min(M, m_begin + p.pixels_per_split);
  double accd[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) accd[i][j] = 0.0;
  // staging: thread -> (pixel 0..31, 8 consecutive channels)
  const int lp = t >> 3, lc = (t & 7) * 8;
  for (long long mb = m_begin; mb < m_end; mb += kF32BK) {
    const long long m = mb + lp;
    float a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, b[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (m < m_end) {
      const int x = (int)(m % p.ow), y = (int)((m / p.ow) % p.oh), bi = (int)(m / ((long long)p.ow * p.oh));
      if (n0 + lc < p.N) {
        const float* src = p.dy + bi * p.dsb + y * p.dsy + x * p.dsx + n0 + lc;
        const float4 u0 = *reinterpret_cast<const float4*>(src);
        a[0] = u0.x; a[1] = u0.y; a[2] = u0.z; a[3] = u0.w;
        if (n0 + lc + 4 < p.N) {
          const float4 u1 = *reinterpret_cast<const float4*>(src + 4);
          a[4] = u1.x; a[5] = u1.y; a[6] = u1.z; a[7] = u1.w;
        }
      }
      const int yy = y + p.tap_dy[tap], xx = x + p.tap_dx[tap];
      if (yy >= 0 && yy < p.vh[v] && xx >= 0 && xx < p.vw[v] && c0 + lc < p.C) {
        const float* src = p.view[v] + bi * p.vsb[v] + yy * p.vsy[v] + xx * p.vsx[v] + c0 + lc;
        const float4 u0 = *reinterpret_cast<const float4*>(src);
        b[0] = u0.x; b[1] = u0.y; b[2] = u0.z; b[3] = u0.w;
        if (c0 + lc + 4 < p.C) {
          const float4 u1 = *reinterpret_cast<const float4*>(src + 4);
          b[4] = u1.x; b[5] = u1.y; b[6] = u1.z; b[7] = u1.w;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { As[lp][lc + j] = a[j]; Bs[lp][lc + j] = b[j]; }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll
    for (int k = 0; k < kF32BK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float aa[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) accd[i][j] += (double)acc[i][j];
    __syncthreads();
  }
  const long long row_len = (long long)p.num_taps * p.C;
  float* dst = p.partial + (long long)blockIdx.z * p.N * row_len;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= p.N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + tx * 4 + j;
      if (c < p.C) dst[n * row_len + (long long)tap * p.C + c] = (float)accd[i][j];
    }
  }
}

__global__ void __launch_bounds__(256) sum_splits_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                                         int splits, long long n, int accumulate) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double t = 0.0;
    for (int s = 0; s < splits; ++s) t += (double)partial[(long long)s * n + i];
    if (accumulate) t += (double)out[i];
    out[i] = (float)t;
  }
}

int conv_wgrad_f32(const odb_wgrad_desc* d, cudaStream_t stream) {
  WgradF32Params p;
  memset(&p, 0, sizeof(p));
  p.C = d->views[0].c;
  if (p.C % 8 != 0 || d->n % 8 != 0) return fail(ODB_ERR_INVALID, "conv_wgrad (fp32 mode): C and n must be multiples of 8");
  for (int v = 0; v < d->num_views; ++v) {
    if (!view_ok(d->views[v]) || d->views[v].c != p.C) return fail(ODB_ERR_INVALID, "conv_wgrad (fp32 mode): bad view");
    p.view[v] = static_cast<const float*>(d->views[v].ptr);
    p.vw[v] = d->views[v].w; p.vh[v] = d->views[v].h;
    fill_strides(d->views[v], &p.vsx[v], &p.vsy[v], &p.vsb[v]);
  }
  p.num_taps = d->num_taps;
  for (int t = 0; t < d->num_taps; ++t) { p.tap_view[t] = d->tap_view[t]; p.tap_dx[t] = d->tap_dx[t]; p.tap_dy[t] = d->tap_dy[t]; }
  if (!view_ok(d->dy) || d->dy.c != d->n) return fail(ODB_ERR_INVALID, "conv_wgrad (fp32 mode): bad dy view");
  p.dy = static_cast<const float*>(d->dy.ptr);
  fill_strides(d->dy, &p.dsx, &p.dsy, &p.dsb);
  p.N = d->n; p.ow = d->dy.w; p.oh = d->dy.h; p.ob = d->dy.b;
  const long long M = (long long)p.ob * p.oh * p.ow;
  const long long row_len = (long long)p.num_taps * p.C;
  const long long tiles = (long long)((p.N + 63) / 64) * ((p.C + 63) / 64) * p.num_taps;
  long long splits = (4LL * num_sms() + tiles - 1) / tiles;
  const long long max_splits = (M + 255) / 256;
  if (splits > max_splits) splits = max_splits;
  if (splits > 256) splits = 256;
  if (splits < 1) splits = 1;
  if ((long long)d->workspace_bytes < splits * p.N * row_len * 4) {
    splits = d->workspace_bytes / (p.N * row_len * 4);
    if (splits < 1) return fail(ODB_ERR_INVALID, "conv_wgrad (fp32 mode): workspace too small (need >= n * taps * C * 4 bytes)");
  }
  p.pixels_per_split = ((M + splits - 1) / splits + kF32BK - 1) / kF32BK * kF32BK;
  p.partial = static_cast<float*>(d->workspace);
  dim3 grid((p.N + 63) / 64, ((p.C + 63) / 64) * p.num_taps, (unsigned)splits);
  wgrad_f32_kernel<<<grid, 256, 0, stream>>>(p);
  count_launch();
  const long long total = p.N * row_len;
  long long blocks = (total + 255) / 256;
  if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
  sum_splits_kernel<<<(unsigned)blocks, 256, 0, stream>>>(p.partial, d->out, (int)splits, total, d->accumulate);
  count_launch();
  return check_launch("conv_wgrad (fp32 mode)");
}

// ---- attention backward, fp32: kernel 1 per (16 queries, head, image): recompute P, dP, dS; write P and dS to the
// workspace and dQ; kernel 2 per (16 keys, head, image): dK = dS^T Q, dV = P^T dO.
__global__ void __launch_bounds__(256) attention_bwd_q_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ o,
                                                                  const float* __restrict__ d_o, float* __restrict__ dqkv,
                                                                  float* __restrict__ pws, float* __restrict__ dsws,
                                                                  int tokens, int heads, float scale) {
  extern __shared__ float att_smem[];
  float (*q_s)[64] = reinterpret_cast<float (*)[64]>(att_smem);
  float (*do_s)[64] = reinterpret_cast<float (*)[64]>(att_smem + kAttQ * 64);
  float (*s_s)[kAttMaxTok] = reinterpret_cast<float (*)[kAttMaxTok]>(att_smem + 2 * kAttQ * 64);                 // S -> P
  float (*g_s)[kAttMaxTok] = reinterpret_cast<float (*)[kAttMaxTok]>(att_smem + 2 * kAttQ * 64 + kAttQ * kAttMaxTok);  // dP -> dS
  float* dd_s = att_smem + 2 * kAttQ * 64 + 2 * kAttQ * kAttMaxTok;
  const int t = threadIdx.x;
  const int q0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const long long rs = 3LL * heads * 64;
  const float* base = qkv + (long long)b * tokens * rs + h * 64;
  const long long orow = (long long)heads * 64;
  for (int i = t; i < kAttQ * 64; i += 256) {
    const int r = i >> 6, d = i & 63;
    const bool ok = q0 + r < tokens;
    q_s[r][d] = ok ? base[(long long)(q0 + r) * rs + d] : 0.f;
    do_s[r][d] = ok ? d_o[((long long)b * tokens + q0 + r) * orow + h * 64 + d] : 0.f;
  }
  __syncthreads();
  if (t < kAttQ) {
    double acc = 0.0;
    if (q0 + t < tokens)
      for (int d = 0; d < 64; ++d) acc += (double)do_s[t][d] * (double)o[((long long)b * tokens + q0 + t) * orow + h * 64 + d];
    dd_s[t] = (float)acc;
  }
  for (int idx = t; idx < kAttQ * tokens; idx += 256) {
    const int r = idx & (kAttQ - 1), j = idx / kAttQ;
    const float* kr = base + (long long)j * rs + heads * 64;
    const float* vr = base + (long long)j * rs + 2 * heads * 64;
    double a = 0.0, g = 0.0;
#pragma unroll 16
    for (int d = 0; d < 64; ++d) { a += (double)q_s[r][d] * (double)kr[d]; g += (double)do_s[r][d] * (double)vr[d]; }
    s_s[r][j] = (float)a * scale;
    g_s[r][j] = (float)g;
  }
  __syncthreads();
  const int warp = t >> 5, lane = t & 31;
  for (int r = warp; r < kAttQ; r += 8) {
    float mx = -INFINITY;
    for (int j = lane; j < tokens; j += 32) mx = fmaxf(mx, s_s[r][j]);
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    double sum = 0.0;
    for (int j = lane; j < tokens; j += 32) { const float e = expf(s_s[r][j] - mx); s_s[r][j] = e; sum += (double)e; }
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
    const float inv = (float)(1.0 / sum);
    const float dd = dd_s[r];
    const bool ok = q0 + r < tokens;
    float* prow = pws + (((long long)b * heads + h) * tokens + q0 + r) * tokens;
    float* drow = dsws + (((long long)b * heads + h) * tokens + q0 + r) * tokens;
    for (int j = lane; j < tokens; j += 32) {
      const float pj = s_s[r][j] * inv;
      const float ds = pj * (g_s[r][j] - dd) * scale;
      g_s[r][j] = ds;
      if (ok) { prow[j] = pj; drow[j] = ds; }
    }
  }
  __syncthreads();
  const int r = t >> 4, d4 = (t & 15) * 4;
  if (q0 + r < tokens) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    const float* kb = base + heads * 64 + d4;
    for (int j = 0; j < tokens; ++j) {
      const double ds = (double)g_s[r][j];
      const float4 kv = *reinterpret_cast<const float4*>(kb + (long long)j * rs);
      a0 += ds * (double)kv.x; a1 += ds * (double)kv.y; a2 += ds * (double)kv.z; a3 += ds * (double)kv.w;
    }
    float* dst = dqkv + ((long long)b * tokens + q0 + r) * rs + h * 64 + d4;
    *reinterpret_cast<float4*>(dst) = make_float4((float)a0, (float)a1, (float)a2, (float)a3);
  }
}

__global__ void __launch_bounds__(256) attention_bwd_kv_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ d_o,
                                                                   const float* __restrict__ pws, const float* __restrict__ dsws,
                                                                   float* __restrict__ dqkv, int tokens, int heads) {
  // thread -> (key row r of 16, 4 head dims)
  const int t = threadIdx.x;
  const int j0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const int r = t >> 4, d4 = (t & 15) * 4;
  const int j = j0 + r;
  if (j >= tokens) return;
  const long long rs = 3LL * heads * 64, orow = (long long)heads * 64;
  const float* qb = qkv + (long long)b * tokens * rs + h * 64 + d4;
  const float* dob = d_o + (long long)b * tokens * orow + h * 64 + d4;
  const float* pcol = pws + ((long long)b * heads + h) * tokens * tokens + j;
  const float* dcol = dsws + ((long long)b * heads + h) * tokens * tokens + j;
  double k0 = 0, k1 = 0, k2 = 0, k3 = 0, v0 = 0, v1 = 0, v2 = 0, v3 = 0;
  for (int q = 0; q < tokens; ++q) {
    const double ds = (double)dcol[(long long)q * tokens], pj = (double)pcol[(long long)q * tokens];
    const float4 qv = *reinterpret_cast<const float4*>(qb + (long long)q * rs);
    const float4 dv = *reinterpret_cast<const float4*>(dob + (long long)q * orow);
    k0 += ds * (double)qv.x; k1 += ds * (double)qv.y; k2 += ds * (double)qv.z; k3 += ds * (double)qv.w;
    v0 += pj * (double)dv.x; v1 += pj * (double)dv.y; v2 += pj * (double)dv.z; v3 += pj * (double)dv.w;
  }
  float* dk = dqkv + ((long long)b * tokens + j) * rs + heads * 64 + h * 64 + d4;
  float* dv_ = dqkv + ((long long)b * tokens + j) * rs + 2 * heads * 64 + h * 64 + d4;
  *reinterpret_cast<float4*>(dk) = make_float4((float)k0, (float)k1, (float)k2, (float)k3);
  *reinterpret_cast<float4*>(dv_) = make_float4((float)v0, (float)v1, (float)v2, (float)v3);
}

int attention_bwd_f32(const float* qkv, const float* o, const float* d_o, float* dqkv, void* workspace,
                      long long workspace_bytes, int b, int tokens, int heads, float scale, cudaStream_t stream) {
  const long long need = 2LL * b * heads * tokens * tokens * 4;
  if (workspace == nullptr || workspace_bytes < need) return fail(ODB_ERR_INVALID, "attention_bwd (fp32 mode): workspace too small");
  if (tokens > kAttMaxTok) return fail(ODB_ERR_UNSUPPORTED, "attention_bwd (fp32 mode): at most 640 tokens");
  float* pws = static_cast<float*>(workspace);
  float* dsws = pws + (long long)b * heads * tokens * tokens;
  dim3 grid((tokens + kAttQ - 1) / kAttQ, heads, b);
  static bool configured[kMaxDevices] = {};
  const int dev = current_device();
  constexpr int kSmem = (2 * kAttQ * 64 + 2 * kAttQ * kAttMaxTok + kAttQ) * 4;
  if (!configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(attention_bwd_q_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return fail_cuda(e, "attention_bwd (fp32 mode): cudaFuncSetAttribute");
    configured[dev] = true;
  }
  attention_bwd_q_f32_kernel<<<grid, 256, kSmem, stream>>>(qkv, o, d_o, dqkv, pws, dsws, tokens, heads, scale);
  count_launch();
  attention_bwd_kv_f32_kernel<<<grid, 256, 0, stream>>>(qkv, d_o, pws, dsws, dqkv, tokens, heads);
  count_launch();
  return check_launch("attention_bwd (fp32 mode)");
}

}  // namespace odb
