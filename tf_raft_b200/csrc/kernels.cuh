// CUDA-core kernels of the RAFT hot path: pyramid lookup (HBM gather), convex upsampling, the fp32
// FFMA contraction path (correlation GEMM, generic NHWC convolution), GRU gating, hi/lo splitting,
// weight re-layout.  All NHWC, fp32 unless a __half plane is named.
#pragma once
#include "common.cuh"

namespace raft {

// ------------------------------------------------------------------------------------------------
// fp32 plane -> fp16 hi/lo planes (operand format of the tensor-core path)
//   src (npix, src_stride) channels [src_c0, src_c0+nch)  ->  hi/lo (npix, dst_stride) at dst_c0;
//   channels [nch, nch_pad) of the destination are written as zeros.
// ------------------------------------------------------------------------------------------------
__global__ void split_plane_kernel(const float* __restrict__ src, int src_stride, int src_c0, int nch, int nch_pad,
                                   __half* __restrict__ hi, __half* __restrict__ lo, int dst_stride, int dst_c0,
                                   size_t npix, float scale) {
  const size_t total = npix * (size_t)nch_pad;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t px = i / nch_pad;
    const int c = (int)(i - px * nch_pad);
    __half h = __float2half_rn(0.f), l = h;
    if (c < nch) split_f16(src[px * src_stride + src_c0 + c] * scale, h, l);
    hi[px * dst_stride + dst_c0 + c] = h;
    lo[px * dst_stride + dst_c0 + c] = l;
  }
}

// 2x2 mean, VALID (floors odd dims), over the two spatial dims of (M, H, W, C) -> (M, H/2, W/2, C).
// Used on the correlation volume (C = 1, corr.py:113) and, by linearity, on fmap2 (C = 256).
__global__ void avgpool2x2_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t M, int H, int W,
                                  int C) {
  const int Ho = H / 2, Wo = W / 2;
  const size_t total = M * (size_t)Ho * Wo * C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t t = i;
    const int c = (int)(t % C);
    t /= C;
    const int xo = (int)(t % Wo);
    t /= Wo;
    const int yo = (int)(t % Ho);
    const size_t m = t / Ho;
    const float* s = src + ((m * H + 2 * yo) * W + 2 * xo) * (size_t)C + c;
    const float a = s[0], b = s[C], cc = s[(size_t)W * C], d = s[(size_t)W * C + C];
    dst[i] = __fmul_rn(__fadd_rn(__fadd_rn(a, b), __fadd_rn(cc, d)), 0.25f);
  }
}

// coords_grid (corr.py:72-90)
__global__ void coords_grid_kernel(float* __restrict__ out, int B, int h, int w) {
  const size_t total = (size_t)B * h * w;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % w), y = (int)((i / w) % h);
    out[2 * i] = (float)x;
    out[2 * i + 1] = (float)y;
  }
}

// ------------------------------------------------------------------------------------------------
// bilinear_sampler (corr.py:28-69), one sample.  floor/ceil corners: an integer (or clamped)
// coordinate gives zero weight on all four corners.  Every operation is individually rounded
// (__f*_rn) so the result is bit-identical to the op-by-op NumPy/TF evaluation.
// ------------------------------------------------------------------------------------------------
struct TapGather { float c00, c01, c10, c11; int o00, o01, o10, o11; };
// Corner offsets and weights of one sample (corr.py:40-60), each operation individually rounded.
__device__ __forceinline__ TapGather tap_setup(int H, int W, float px, float py) {
  const float gx = fminf(fmaxf(px, 0.0f), (float)(W - 1));
  const float gy = fminf(fmaxf(py, 0.0f), (float)(H - 1));
  const float gx0 = floorf(gx), gx1 = ceilf(gx), gy0 = floorf(gy), gy1 = ceilf(gy);
  const float wy1 = __fsub_rn(gy1, gy), wy0 = __fsub_rn(gy, gy0);
  const float wx1 = __fsub_rn(gx1, gx), wx0 = __fsub_rn(gx, gx0);
  TapGather t;
  t.c00 = __fmul_rn(wy1, wx1); t.c01 = __fmul_rn(wy1, wx0);
  t.c10 = __fmul_rn(wy0, wx1); t.c11 = __fmul_rn(wy0, wx0);
  const int ix0 = (int)gx0, ix1 = (int)gx1, iy0 = (int)gy0, iy1 = (int)gy1;
  t.o00 = iy0 * W + ix0; t.o01 = iy0 * W + ix1; t.o10 = iy1 * W + ix0; t.o11 = iy1 * W + ix1;
  return t;
}
__device__ __forceinline__ float tap_combine(const TapGather& t, float x00, float x01, float x10, float x11) {
  float acc = __fmul_rn(t.c00, x00);                       // corr.py:68, left to right
  acc = __fadd_rn(acc, __fmul_rn(t.c01, x01));
  acc = __fadd_rn(acc, __fmul_rn(t.c10, x10));
  acc = __fadd_rn(acc, __fmul_rn(t.c11, x11));
  return acc;
}
__device__ __forceinline__ float sample_floor_ceil(const float* __restrict__ img, int H, int W, float px, float py) {
  const TapGather t = tap_setup(H, W, px, py);
  return tap_combine(t, __ldg(img + t.o00), __ldg(img + t.o01), __ldg(img + t.o10), __ldg(img + t.o11));
}

__global__ void bilinear_sampler_kernel(const float* __restrict__ image, const float* __restrict__ coords, int M, int H,
                                        int W, int P, float* __restrict__ out) {
  const size_t total = (size_t)M * P;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t m = i / P;
    out[i] = sample_floor_ceil(image + m * (size_t)H * W, H, W, coords[2 * i], coords[2 * i + 1]);
  }
}

// ------------------------------------------------------------------------------------------------
// CorrBlock.retrieve (corr.py:116-152).  One warp per (query pixel, level); lanes stride over the
// (2r+1)^2 taps, so the output row segment is written coalesced.  Tap t = a*(2r+1)+b has x-offset
// a-r and y-offset b-r (corr.py:133-143).  Optionally also emits the fp16 hi/lo planes the
// tensor-core update block consumes (channels beyond levels*(2r+1)^2 up to h_pad are zeroed).
// ------------------------------------------------------------------------------------------------
struct LookupParams {
  const float* pyr[RAFT_MAX_LEVELS];
  int lh[RAFT_MAX_LEVELS], lw[RAFT_MAX_LEVELS];
  const float* coords;
  float* out; int out_stride;
  __half* out_hi; __half* out_lo; int h_stride, h_pad;
  int nq;      // B*h*w
  int levels, radius;
  // Optional rider of the window kernel (iteration loop): the 7x7 im2col of the current flow for convf1 (update.py:92) --
  // independent of the lookup, tiny, and one launch less per iteration when it shares the lookup's grid.
  const float* im_flow; __half* im_hi; __half* im_lo; int im_B, im_h, im_w;
};

__global__ void __launch_bounds__(256) corr_lookup_kernel(const LookupParams p) {
  __shared__ float4 axis_smem[8 * 32];                          // per warp: 16 x-axis + 16 y-axis tap set-ups
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int side = 2 * p.radius + 1, ntap = side * side;
  const size_t nwork = (size_t)p.nq * p.levels;
  for (size_t wi = (size_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5); wi < nwork;
       wi += (size_t)gridDim.x * warps_per_block) {
    const int q = (int)(wi / p.levels), l = (int)(wi % p.levels);
    const int H = p.lh[l], W = p.lw[l];
    const float* img = p.pyr[l] + (size_t)q * H * W;
    const float inv = 1.0f / (float)(1 << l);                    // exact power of two
    const float cx = __fmul_rn(__ldg(p.coords + 2 * (size_t)q), inv);     // coords / 2**i  (corr.py:141)
    const float cy = __fmul_rn(__ldg(p.coords + 2 * (size_t)q + 1), inv);
    // The x-part of a tap depends only on a, the y-part only on b: the 2*(2r+1) axis set-ups (clamp, floor, ceil,
    // weights, indices -- corr.py:40-60) are computed once per (query, level) by lanes 0..2*side-1 and shared through
    // shared memory; each tap then only multiplies weights and adds indices -- the same fp32 operations in the same
    // order as the per-tap evaluation, so results stay bit-identical.  All gathers are issued before any is consumed
    // (the kernel is latency / instruction bound, not bandwidth bound).
    constexpr int kMaxIter = 3;                                  // (2r+1)^2 <= 96, i.e. radius <= 4
    if (ntap <= 32 * kMaxIter && side <= 16) {
      float4* ax = axis_smem + (threadIdx.x >> 5) * 32;          // [0,16): x set-ups, [16,32): y set-ups
      __syncwarp();
      if (lane < 2 * side) {
        const bool isy = lane >= side;
        const int i = isy ? lane - side : lane;
        const float cc = isy ? cy : cx;
        const int dim = isy ? H : W;
        const float g = fminf(fmaxf(__fadd_rn(cc, (float)(i - p.radius)), 0.0f), (float)(dim - 1));   // centroid + delta, clamp
        const float g0 = floorf(g), g1 = ceilf(g);
        ax[(isy ? 16 : 0) + i] = make_float4(__fsub_rn(g1, g), __fsub_rn(g, g0), __int_as_float((int)g0), __int_as_float((int)g1));
      }
      __syncwarp();
      TapGather tg[kMaxIter];
      float x00[kMaxIter], x01[kMaxIter], x10[kMaxIter], x11[kMaxIter];
#pragma unroll
      for (int i = 0; i < kMaxIter; ++i) {
        const int t = min(lane + 32 * i, ntap - 1);
        const int a = t / side, b2 = t - a * side;
        const float4 sx = ax[a], sy = ax[16 + b2];               // (w1, w0, i0, i1) per axis
        const int ix0 = __float_as_int(sx.z), ix1 = __float_as_int(sx.w), iy0 = __float_as_int(sy.z), iy1 = __float_as_int(sy.w);
        tg[i].c00 = __fmul_rn(sy.x, sx.x); tg[i].c01 = __fmul_rn(sy.x, sx.y);
        tg[i].c10 = __fmul_rn(sy.y, sx.x); tg[i].c11 = __fmul_rn(sy.y, sx.y);
        x00[i] = __ldg(img + iy0 * W + ix0); x01[i] = __ldg(img + iy0 * W + ix1);
        x10[i] = __ldg(img + iy1 * W + ix0); x11[i] = __ldg(img + iy1 * W + ix1);
      }
#pragma unroll
      for (int i = 0; i < kMaxIter; ++i) {
        const int t = lane + 32 * i;
        if (t < ntap) {
          const float v = tap_combine(tg[i], x00[i], x01[i], x10[i], x11[i]);
          const int ch = l * ntap + t;
          if (p.out) p.out[(size_t)q * p.out_stride + ch] = v;
          if (p.out_hi) {
            __half hh, ll;
            split_f16(v, hh, ll);
            p.out_hi[(size_t)q * p.h_stride + ch] = hh;
            p.out_lo[(size_t)q * p.h_stride + ch] = ll;
          }
        }
      }
    } else {
      for (int t = lane; t < ntap; t += 32) {
        const int a = t / side, b2 = t - a * side;
        const float px = __fadd_rn(cx, (float)(a - p.radius));   // centroid + delta (corr.py:143)
        const float py = __fadd_rn(cy, (float)(b2 - p.radius));
        const float v = sample_floor_ceil(img, H, W, px, py);
        const int ch = l * ntap + t;
        if (p.out) p.out[(size_t)q * p.out_stride + ch] = v;
        if (p.out_hi) {
          __half hh, ll;
          split_f16(v, hh, ll);
          p.out_hi[(size_t)q * p.h_stride + ch] = hh;
          p.out_lo[(size_t)q * p.h_stride + ch] = ll;
        }
      }
    }
    if (p.out_hi && l == p.levels - 1) {
      const __half zero = __float2half_rn(0.f);
      for (int c = p.levels * ntap + lane; c < p.h_pad; c += 32) {
        p.out_hi[(size_t)q * p.h_stride + c] = zero;
        p.out_lo[(size_t)q * p.h_stride + c] = zero;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 correlation (RAFT_PREC_FP32): out[b, q, n] = <f1[b,q,:], f2[b,n,:]> / sqrt(C)  (corr.py:154-162)
// 64x64 tile, 16-wide K slab, 4x4 micro-tile per thread.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) corr_fp32_kernel(const float* __restrict__ f1, const float* __restrict__ f2,
                                                        float* __restrict__ out, int N, int C, float div) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int b = blockIdx.z;
  const float* A = f1 + (size_t)b * N * C;
  const float* Bm = f2 + (size_t)b * N * C;
  float* O = out + (size_t)b * N * N;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lr = threadIdx.x >> 2, lc = (threadIdx.x & 3) * 4;   // loader: row 0..63, 4 consecutive k
  float acc[4][4] = {};
  for (int k0 = 0; k0 < C; k0 += 16) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + lc + j;
      As[lc + j][lr] = (m0 + lr < N && k < C) ? A[(size_t)(m0 + lr) * C + k] : 0.f;
      Bs[lc + j][lr] = (n0 + lr < N && k < C) ? Bm[(size_t)(n0 + lr) * C + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a[i] = As[k][ty * 4 + i];
        w[i] = Bs[k][tx * 4 + i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < N && n < N) O[(size_t)m * N + n] = __fdiv_rn(acc[i][j], div);
    }
}

// ------------------------------------------------------------------------------------------------
// Generic stride-1 'same' convolution, fp32 FFMA (RAFT_PREC_FP32 path and the Cin=2 7x7 flow conv
// of the tensor-core path).  Input = channel concat of up to 3 NHWC sources; HWIO weights.
//   out[pix, c0+n] = act(bias[n] + sum_{tap,c} in[pix+tap, c] * w[tap, c, n]) * out_scale
// 64 px x 64 cout tile, 16-channel slab per tap, 4x4 micro-tile per thread.
// ------------------------------------------------------------------------------------------------
enum SimtAct : int { SACT_NONE = 0, SACT_RELU = 1, SACT_SIGMOID = 2, SACT_TANH = 3 };

struct SimtConvParams {
  const float* src[3]; int src_stride[3], src_c0[3], src_n[3]; int nsrc;
  const float* w; const float* bias;         // HWIO (kh, kw, cin, cout)
  int kh, kw, cin, cout;
  int B, H, W;                               // OUTPUT grid
  int stride, Hin, Win, pad_t, pad_l;        // stride 0/1 => stride 1, input grid = output grid, symmetric 'same' pads
  int in_image_norm;                         // 1: input is a 0..255 image, normalised on load as 2*(x/255)-1 (model.py:70-71)
  const float* post_scale; const float* post_shift;   // optional per-cout affine after the bias (folded BatchNorm)
  float* out; int out_stride, out_c0;
  __half* out_hi; __half* out_lo; int h_stride, h_c0;   // optional fp16 hi/lo copy of the output
  int act; float out_scale;
};

__global__ void __launch_bounds__(256) conv_simt_kernel(const SimtConvParams p) {
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int npix = p.B * p.H * p.W;
  const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lr = threadIdx.x >> 2, lc = (threadIdx.x & 3) * 4;   // A loader: pixel row, 4 channels
  const int wr = threadIdx.x >> 4, wc = (threadIdx.x & 15) * 4;  // W loader: k row, 4 couts
  const int st = p.stride > 1 ? p.stride : 1;
  const int Hin = p.stride > 0 ? p.Hin : p.H, Win = p.stride > 0 ? p.Win : p.W;
  const int ph = p.stride > 0 ? p.pad_t : (p.kh - 1) / 2, pw = p.stride > 0 ? p.pad_l : (p.kw - 1) / 2;
  // this thread's loader pixel
  const int lp = m0 + lr;
  int lb = 0, ly = 0, lx = 0;
  if (lp < npix) {
    lx = lp % p.W;
    ly = (lp / p.W) % p.H;
    lb = lp / (p.W * p.H);
  }
  float acc[4][4] = {};
  for (int tap = 0; tap < p.kh * p.kw; ++tap) {
    const int dy = tap / p.kw - ph, dx = tap % p.kw - pw;
    const int sy = ly * st + dy, sx = lx * st + dx;
    const bool inb = lp < npix && sy >= 0 && sy < Hin && sx >= 0 && sx < Win;
    const size_t spix = ((size_t)lb * Hin + (inb ? sy : 0)) * Win + (inb ? sx : 0);
    for (int k0 = 0; k0 < p.cin; k0 += 16) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = k0 + lc + j;
        float v = 0.f;
        if (inb && c < p.cin) {
          int cc = c, s = 0;
          while (s < p.nsrc - 1 && cc >= p.src_n[s]) cc -= p.src_n[s++];
          v = __ldg(p.src[s] + spix * p.src_stride[s] + p.src_c0[s] + cc);
          if (p.in_image_norm) v = __fsub_rn(__fmul_rn(2.0f, __fdiv_rn(v, 255.0f)), 1.0f);
        }
        As[lc + j][lr] = v;
      }
      {
        const int c = k0 + wr;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = n0 + wc + j;
          Ws[wr][wc + j] = (c < p.cin && n < p.cout) ? __ldg(p.w + ((size_t)tap * p.cin + c) * p.cout + n) : 0.f;
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        float a[4], w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          a[i] = As[k][ty * 4 + i];
          w[i] = Ws[k][tx * 4 + i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= npix) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.cout) continue;
      float v = acc[i][j] + (p.bias ? __ldg(p.bias + n) : 0.f);
      if (p.post_scale) v = v * __ldg(p.post_scale + n) + __ldg(p.post_shift + n);
      if (p.act == SACT_RELU) v = fmaxf(v, 0.f);
      else if (p.act == SACT_SIGMOID) v = sigmoidf_acc(v);
      else if (p.act == SACT_TANH) v = tanhf(v);
      v *= p.out_scale;
      if (p.out) p.out[(size_t)m * p.out_stride + p.out_c0 + n] = v;
      if (p.out_hi) {
        __half hh, ll;
        split_f16(v, hh, ll);
        p.out_hi[(size_t)m * p.h_stride + p.h_c0 + n] = hh;
        p.out_lo[(size_t)m * p.h_stride + p.h_c0 + n] = ll;
      }
    }
  }
}

// GRU gating (update.py:32-34, 55-66), fp32 path.
__global__ void gru_rh_kernel(const float* __restrict__ r, const float* __restrict__ h, float* __restrict__ rh,
                              size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    rh[i] = r[i] * h[i];
}
__global__ void gru_update_kernel(const float* __restrict__ z, const float* __restrict__ q, float* __restrict__ h,
                                  size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    h[i] = (1.0f - z[i]) * h[i] + z[i] * q[i];
}

// Strided channel copy: dst[px, dst_c0 + c] = src[px, src_c0 + c], c < n.
__global__ void copy_channels_kernel(const float* __restrict__ src, int src_stride, int src_c0,
                                     float* __restrict__ dst, int dst_stride, int dst_c0, int n, size_t npix) {
  const size_t total = npix * (size_t)n;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t px = i / n;
    const int c = (int)(i - px * n);
    dst[px * dst_stride + dst_c0 + c] = src[px * src_stride + src_c0 + c];
  }
}

// model.py:97,102: coords1 += delta_flow (in place); flow = coords1 - coords0 with coords0 the
// pixel grid (model.py:89), recomputed from the index instead of being stored.
__global__ void flow_advance_kernel(float* __restrict__ coords1, const float* __restrict__ delta,
                                    float* __restrict__ flow, int B, int h, int w) {
  const size_t total = (size_t)B * h * w;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const float gx = (float)(i % w), gy = (float)((i / w) % h);
    float cx = coords1[2 * i], cy = coords1[2 * i + 1];
    if (delta) {
      cx = __fadd_rn(cx, delta[2 * i]);
      cy = __fadd_rn(cy, delta[2 * i + 1]);
      coords1[2 * i] = cx;
      coords1[2 * i + 1] = cy;
    }
    flow[2 * i] = __fsub_rn(cx, gx);
    flow[2 * i + 1] = __fsub_rn(cy, gy);
  }
}

// ------------------------------------------------------------------------------------------------
// RAFT.upsample_flow (model.py:39-66): one 64-thread group per coarse pixel, thread = (by, bx).
// mask channel (by*8+bx)*9 + ky*3+kx; softmax over the 9 taps; neighbours of 8*flow zero-padded.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upsample_convex_kernel(const float* __restrict__ flow,
                                                              const float* __restrict__ mask, int B, int h, int w,
                                                              float* __restrict__ out) {
  const int sub = threadIdx.x & 63;
  const size_t npix = (size_t)B * h * w;
  for (size_t pix = (size_t)blockIdx.x * 4 + (threadIdx.x >> 6); pix < npix; pix += (size_t)gridDim.x * 4) {
    const int x = (int)(pix % w), y = (int)((pix / w) % h), b = (int)(pix / ((size_t)w * h));
    const float* mp = mask + pix * 576 + sub * 9;
    float m[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      m[k] = __ldg(mp + k);
      mx = fmaxf(mx, m[k]);
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      m[k] = expf(m[k] - mx);
      sum += m[k];
    }
    float ox = 0.f, oy = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int yy = y + k / 3 - 1, xx = x + k % 3 - 1;
      float fx = 0.f, fy = 0.f;
      if (yy >= 0 && yy < h && xx >= 0 && xx < w) {
        const float* fp = flow + (((size_t)b * h + yy) * w + xx) * 2;
        fx = 8.0f * __ldg(fp);
        fy = 8.0f * __ldg(fp + 1);
      }
      const float wk = m[k] / sum;
      ox += wk * fx;
      oy += wk * fy;
    }
    const int by = sub >> 3, bx = sub & 7;
    float* op = out + ((((size_t)b * 8 * h) + 8 * y + by) * (8 * (size_t)w) + 8 * x + bx) * 2;
    *reinterpret_cast<float2*>(op) = make_float2(ox, oy);
  }
}

// upflow8 (corr.py:93-96): 8 * bilinear resize, half-pixel centres, edge-clamped source indices.
__global__ void upflow8_kernel(const float* __restrict__ flow, int B, int h, int w, float* __restrict__ out) {
  const int H = 8 * h, W = 8 * w;
  const size_t total = (size_t)B * H * W;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % W), Y = (int)((i / W) % H), b = (int)(i / ((size_t)W * H));
    const float sx = ((float)X + 0.5f) * 0.125f - 0.5f, sy = ((float)Y + 0.5f) * 0.125f - 0.5f;
    const float fx0 = floorf(sx), fy0 = floorf(sy);
    const float ax = sx - fx0, ay = sy - fy0;
    const int x0 = min(max((int)fx0, 0), w - 1), x1 = min(max((int)fx0 + 1, 0), w - 1);
    const int y0 = min(max((int)fy0, 0), h - 1), y1 = min(max((int)fy0 + 1, 0), h - 1);
    const float* f = flow + (size_t)b * h * w * 2;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float v00 = f[((size_t)y0 * w + x0) * 2 + c], v01 = f[((size_t)y0 * w + x1) * 2 + c];
      const float v10 = f[((size_t)y1 * w + x0) * 2 + c], v11 = f[((size_t)y1 * w + x1) * 2 + c];
      const float top = v00 * (1.f - ax) + v01 * ax, bot = v10 * (1.f - ax) + v11 * ax;
      out[2 * i + c] = 8.0f * (top * (1.f - ay) + bot * ay);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Weight re-layout for the tensor-core path.
//   HWIO fp32 (kh,kw,cin,cout)  ->  [tap][cout_pad][cin_pad] fp16 hi / lo planes of w * 2^k,
//   placed at (cout_off, cin remapped through up to two ranges).  2^k is chosen so that
//   max|w|*2^k lies in [2^12, 2^13): the lo residuals then stay in fp16's normal range.
// ------------------------------------------------------------------------------------------------
__global__ void absmax_kernel(const float* __restrict__ w, size_t n, unsigned int* __restrict__ out_bits) {
  float m = 0.f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(w[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));   // non-negative floats order as uints
}

// scale[0] = 2^k, scale[1] = 2^-k from the absmax bits (shared by all convs merged into one layer)
__global__ void weight_scale_kernel(const unsigned int* __restrict__ absmax_bits, float* __restrict__ scale) {
  const float m = __uint_as_float(*absmax_bits);
  int k = 0;
  if (m > 0.f && isfinite(m)) {
    int e;
    frexpf(m, &e);          // m = f * 2^e, f in [0.5, 1)  ->  m*2^(13-e) in [2^12, 2^13)
    k = 13 - e;
    k = max(-24, min(24, k));
  }
  scale[0] = ldexpf(1.0f, k);
  scale[1] = ldexpf(1.0f, -k);
}

struct PackParams {
  const float* w; int kh, kw, cin, cout;
  __half* hi; __half* lo; int cout_pad, cin_pad, cout_off;
  int r_src0[2], r_n[2], r_dst0[2], nrange;     // cin remap ranges
  const float* scale;                           // scale[0] = 2^k
};
__global__ void pack_weights_kernel(const PackParams p) {
  const size_t total = (size_t)p.kh * p.kw * p.cin * p.cout;
  const float s = p.scale[0];
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t t = i;
    const int n = (int)(t % p.cout);
    t /= p.cout;
    const int c = (int)(t % p.cin);
    const int tap = (int)(t / p.cin);
    int cd = -1;
    for (int r = 0; r < p.nrange; ++r)
      if (c >= p.r_src0[r] && c < p.r_src0[r] + p.r_n[r]) cd = p.r_dst0[r] + (c - p.r_src0[r]);
    if (cd < 0) continue;
    __half hh, ll;
    split_f16(p.w[i] * s, hh, ll);
    const size_t o = ((size_t)tap * p.cout_pad + p.cout_off + n) * p.cin_pad + cd;
    p.hi[o] = hh;
    p.lo[o] = ll;
  }
}

// ------------------------------------------------------------------------------------------------
// Normalisation layers of the encoders (extractor.py:6-16): tfa InstanceNormalization (statistics per
// image) / Keras BatchNormalization in training mode (statistics over the batch), eps = 1e-3.
// y is the raw convolution output (G groups x P pixels x C channels, fp32).  ONE pass over y:
// every thread accumulates shifted sums of its pixels (shift = its first sample, so there is no
// E[x^2]-E[x]^2 cancellation), partial (n, mean, M2) triples are merged with Chan's formula in a fixed
// order (deterministic).   part[g][split][{n, mean, M2}][c]
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void chan_merge(float& na, float& ma, float& m2a, float nb, float mb, float m2b) {
  if (nb == 0.f) return;
  const float n = na + nb, d = mb - ma;
  ma = ma + d * (nb / n);
  m2a = m2a + m2b + d * d * (na * nb / n);
  na = n;
}
// Block (g, split) covers pixels [p0, p1) of group g, per = ceil(P / nsplit).  Within it, lanes = 256 / C pixel lanes
// (lane pl takes pixels p0 + pl, p0 + pl + lanes, ...) and every (lane, channel) sequence is accumulated in pixel order.
// A thread owns one lane and 4 consecutive channels (C % 4 == 0): float4 loads, kNormStatsAhead pixels of its sequence
// loaded before they are summed, so that ~16 MB are in flight over the GPU at G = 8 (the scalar one-channel form kept
// 4 loads per thread in flight and ran latency-bound at ~2.6 TB/s).  The sums, their order and the merge are per channel
// exactly those of a one-thread-per-(lane, channel) loop, so `part` does not depend on this layout.
constexpr int kNormStatsThreads = 64;    // = lanes * C / 4 for C dividing 256 (48 of them work at C = 96)
constexpr int kNormStatsAhead = 32;
__global__ void __launch_bounds__(kNormStatsThreads) norm_stats_kernel(const float* __restrict__ y, int P, int C,
                                                                       int nsplit, float* __restrict__ part) {
  __shared__ float red[3][256];
  const int g = blockIdx.x, sp = blockIdx.y;
  const int lanes = 256 / C > 0 ? 256 / C : 1;          // pixel lanes per split (C <= 256)
  const int cq = C / 4;
  const int c = (threadIdx.x % cq) * 4, pl = threadIdx.x / cq;
  const int per = (P + nsplit - 1) / nsplit;
  const int p0 = sp * per, p1 = min(P, p0 + per);
  float n = 0.f, mean[4] = {0.f, 0.f, 0.f, 0.f}, m2[4] = {0.f, 0.f, 0.f, 0.f};
  if (pl < lanes && p0 + pl < p1) {
    const float4* q = reinterpret_cast<const float4*>(y + ((size_t)g * P + p0 + pl) * C + c);
    const size_t step = (size_t)lanes * cq;             // float4s from one sample of the sequence to the next
    const int cnt = (p1 - p0 - pl + lanes - 1) / lanes;
    const float4 k4 = __ldg(q);                         // shift = the first sample
    const float K[4] = {k4.x, k4.y, k4.z, k4.w};
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = 0; i < cnt; i += kNormStatsAhead) {
      float4 b[kNormStatsAhead];
#pragma unroll
      for (int u = 0; u < kNormStatsAhead; ++u)
        if (i + u < cnt) b[u] = __ldg(q + (size_t)(i + u) * step);
#pragma unroll
      for (int u = 0; u < kNormStatsAhead; ++u) {
        if (i + u < cnt) {
          const float x[4] = {b[u].x, b[u].y, b[u].z, b[u].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v = x[e] - K[e];
            s1[e] += v;
            s2[e] = __fmaf_rn(v, v, s2[e]);             // s2 += v * v, one rounding (FFMA)
          }
          n += 1.f;
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      mean[e] = K[e] + s1[e] / n;
      m2[e] = fmaxf(s2[e] - s1[e] * s1[e] / n, 0.f);
    }
  }
  if (pl < lanes) {
#pragma unroll
    for (int e = 0; e < 4; ++e) { red[0][pl * C + c + e] = n; red[1][pl * C + c + e] = mean[e]; red[2][pl * C + c + e] = m2[e]; }
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < C; ch += kNormStatsThreads) {     // merge lanes 1..lanes-1 into lane 0, in order
    float nn = red[0][ch], mm = red[1][ch], mq = red[2][ch];
    for (int l = 1; l < lanes; ++l) chan_merge(nn, mm, mq, red[0][l * C + ch], red[1][l * C + ch], red[2][l * C + ch]);
    float* o = part + (((size_t)g * nsplit + sp) * 3) * C + ch;
    o[0] = nn; o[C] = mm; o[2 * C] = mq;
  }
}
// mean[g][c] and mult[g][c] = rsqrt(var + eps) * gamma[c]  (the multiplier applied to (y - mean)).
// One warp per (g, c): lanes merge their partials, then a fixed xor-shuffle tree (deterministic).
__global__ void norm_final_kernel(const float* __restrict__ part, int G, int C, int nsplit,
                                  const float* __restrict__ gamma, float eps, float* __restrict__ mean_out,
                                  float* __restrict__ mult_out) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= G * C) return;
  const int g = i / C, c = i % C;
  float n = 0.f, mean = 0.f, m2 = 0.f;
  for (int s = lane; s < nsplit; s += 32) {
    const float* o = part + (((size_t)g * nsplit + s) * 3) * C + c;
    chan_merge(n, mean, m2, o[0], o[C], o[2 * C]);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float nb = __shfl_xor_sync(0xffffffffu, n, off), mb = __shfl_xor_sync(0xffffffffu, mean, off),
                m2b = __shfl_xor_sync(0xffffffffu, m2, off);
    // both partners compute the same merged triple (merge in lane order so the result is bitwise identical)
    float na = n, ma = mean, m2a = m2;
    if (lane & off) { na = nb; ma = mb; m2a = m2b; chan_merge(na, ma, m2a, n, mean, m2); }
    else chan_merge(na, ma, m2a, nb, mb, m2b);
    n = na; mean = ma; m2 = m2a;
  }
  if (lane == 0) {
    mean_out[i] = mean;
    mult_out[i] = rsqrtf(m2 / n + eps) * gamma[c];
  }
}
// out = [relu]((y - mean) * a + beta);  optional skip: out = relu(skip + out)  (ResBlock, extractor.py:41-49)
// skip comes either as an fp32 plane (skip32, C channels) or as the fp16 hi/lo operand planes of the block input
// (skip_hi/lo, c_pad channels; hi + lo reproduces the fp32 value to 2^-23).  Writes fp32 (optional) and the fp16
// hi/lo operand planes (optional; channels [C, c_pad) zeroed).  One thread = 8 consecutive channels (C % 8 == 0).
__global__ void norm_apply_kernel(const float* __restrict__ y, size_t npix, int P, int C, int per_image,
                                  const float* __restrict__ mean, const float* __restrict__ a,
                                  const float* __restrict__ beta, int relu, const float* __restrict__ skip32,
                                  const __half* __restrict__ skip_hi, const __half* __restrict__ skip_lo,
                                  float* __restrict__ out32, __half* __restrict__ hi, __half* __restrict__ lo,
                                  int c_pad) {
  const int gpp = c_pad >> 3;                                    // 8-channel groups per pixel
  const size_t total = npix * (size_t)gpp;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t px = i / gpp;
    const int c = (int)(i - px * gpp) << 3;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c < C) {
      const size_t g = per_image ? px / P : 0;
      const float* yp = y + px * C + c;
      const float* mp = mean + g * C + c;
      const float* ap = a + g * C + c;
      const float* bp = beta + c;
      float4 t[2] = {*reinterpret_cast<const float4*>(yp), *reinterpret_cast<const float4*>(yp + 4)};
      const float yy[8] = {t[0].x, t[0].y, t[0].z, t[0].w, t[1].x, t[1].y, t[1].z, t[1].w};
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[e] = (yy[e] - __ldg(mp + e)) * __ldg(ap + e) + __ldg(bp + e);
        if (relu) v[e] = fmaxf(v[e], 0.f);
      }
      if (skip32) {
        const float4 s0 = *reinterpret_cast<const float4*>(skip32 + px * C + c), s1 = *reinterpret_cast<const float4*>(skip32 + px * C + c + 4);
        const float ss[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = fmaxf(ss[e] + v[e], 0.f);
      } else if (skip_hi) {
        const uint4 h4 = *reinterpret_cast<const uint4*>(skip_hi + px * c_pad + c), l4 = *reinterpret_cast<const uint4*>(skip_lo + px * c_pad + c);
        const uint32_t hw[4] = {h4.x, h4.y, h4.z, h4.w}, lw[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[e]));
          const float2 lf = __half22float2(*reinterpret_cast<const __half2*>(&lw[e]));
          v[2 * e] = fmaxf(hf.x + lf.x + v[2 * e], 0.f);
          v[2 * e + 1] = fmaxf(hf.y + lf.y + v[2 * e + 1], 0.f);
        }
      }
      if (out32) {
        *reinterpret_cast<float4*>(out32 + px * C + c) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(out32 + px * C + c + 4) = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
    if (hi) {
      uint32_t ph[4], pl[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) split_f16x2(v[2 * e], v[2 * e + 1], ph[e], pl[e]);
      *reinterpret_cast<uint4*>(hi + px * c_pad + c) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
      *reinterpret_cast<uint4*>(lo + px * c_pad + c) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
    }
  }
}
// Stem gather (extractor.py:95, model.py:70-71): for every output pixel of the 7x7 stride-2 'same' convolution,
// the 147 input values (tap-major, then rgb) of its window, optionally normalised 2*(x/255)-1, zero outside the image
// (padding applies to the normalised image), as fp16 hi/lo planes with 192 channels (147..191 = 0).
// A block owns kStemSeg output pixels of one output row.  It first stages the 7 input rows x (2 * kStemSeg + 5) columns
// x rgb its windows cover in shared memory (coalesced, each input value loaded and normalised once per block), then
// writes the planes with one 16-byte store per thread and plane (8 consecutive channels of one pixel).
constexpr int kStemSeg = 128;
constexpr int kStemRow = 3 * (2 * kStemSeg + 5);     // floats of one staged input row
__global__ void __launch_bounds__(256) stem_gather_kernel(const float* __restrict__ img, int H, int W, int h, int w,
                                                          int pad_t, int pad_l, int image_norm, __half* __restrict__ hi,
                                                          __half* __restrict__ lo) {
  __shared__ float tile[7 * kStemRow];
  const int x0 = blockIdx.x * kStemSeg, y = blockIdx.y, n = blockIdx.z;
  const int iy0 = 2 * y - pad_t, ix0 = 2 * x0 - pad_l;
  // tile[ty][3 * (ix - ix0) + rgb]: input row iy0 + ty is contiguous in NHWC from column ix0 on
  constexpr int kPerRow = (kStemRow + 255) / 256;
  float v[7][kPerRow];
#pragma unroll
  for (int ty = 0; ty < 7; ++ty) {
    const int iy = iy0 + ty;
    const float* row = img + (((ptrdiff_t)n * H + iy) * W + ix0) * 3;   // only dereferenced in bounds
#pragma unroll
    for (int k = 0; k < kPerRow; ++k) {
      const int j = threadIdx.x + 256 * k, ix = ix0 + j / 3;
      v[ty][k] = 0.f;
      if (j < kStemRow && iy >= 0 && iy < H && ix >= 0 && ix < W) v[ty][k] = __ldg(row + j);
    }
  }
#pragma unroll
  for (int ty = 0; ty < 7; ++ty) {
    const int iy = iy0 + ty;
#pragma unroll
    for (int k = 0; k < kPerRow; ++k) {
      const int j = threadIdx.x + 256 * k, ix = ix0 + j / 3;
      if (j < kStemRow) {
        float x = v[ty][k];
        if (image_norm && iy >= 0 && iy < H && ix >= 0 && ix < W) x = __fsub_rn(__fmul_rn(2.0f, __fdiv_rn(x, 255.0f)), 1.0f);
        tile[ty * kStemRow + j] = x;
      }
    }
  }
  __syncthreads();
  const int npx = min(kStemSeg, w - x0);
  uint4* ohi = reinterpret_cast<uint4*>(hi) + (((size_t)n * h + y) * w + x0) * 24;
  uint4* olo = reinterpret_cast<uint4*>(lo) + (((size_t)n * h + y) * w + x0) * 24;
  for (int i = threadIdx.x; i < npx * 24; i += 256) {
    const int px = i / 24, grp = i - px * 24;
    uint32_t ph[4] = {0u, 0u, 0u, 0u}, pl[4] = {0u, 0u, 0u, 0u};
    if (grp * 8 < 147) {
      // channel kk = (window row ty) * 21 + j, j = 3 * (window column) + rgb: the window of pixel px starts at column
      // 2 * px of the tile, so its value is tile[ty][6 * px + j]; walk (ty, j) incrementally.
      int ty = (grp * 8) / 21, j = grp * 8 - ty * 21;
      const float* t = tile + 6 * px;
      float f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        f[e] = ty < 7 ? t[ty * kStemRow + j] : 0.f;
        if (++j == 21) { j = 0; ++ty; }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) split_f16x2(f[2 * e], f[2 * e + 1], ph[e], pl[e]);
    }
    ohi[i] = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    olo[i] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
  }
}

// The same gather, 8 channels (4 taps x 2 flow components) per thread and 16-byte stores, as a grid-stride device routine
// (called by every thread of corr_lookup_win_kernel after its lookups when the loop asks for it; values identical to
// flow_im2col_kernel).
__device__ __forceinline__ void flow_im2col_rider(const float* __restrict__ flow, int B, int h, int w, __half* __restrict__ hi,
                                                  __half* __restrict__ lo, size_t tid, size_t nthreads) {
  const size_t total = (size_t)B * h * w * 16;
  for (size_t i = tid; i < total; i += nthreads) {
    const int g = (int)(i & 15);
    const size_t px = i >> 4;
    const int x = (int)(px % w), y = (int)((px / w) % h);
    uint32_t ph[4], pl[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int tap = 4 * g + e;
      float2 v = make_float2(0.f, 0.f);
      if (tap < 49) {
        const int yy = y + tap / 7 - 3, xx = x + tap % 7 - 3;
        if (yy >= 0 && yy < h && xx >= 0 && xx < w)
          v = __ldg(reinterpret_cast<const float2*>(flow) + (ptrdiff_t)px + (ptrdiff_t)(yy - y) * w + (xx - x));
      }
      split_f16x2(v.x, v.y, ph[e], pl[e]);
    }
    reinterpret_cast<uint4*>(hi)[i] = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    reinterpret_cast<uint4*>(lo)[i] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
  }
}

// im2col of the 7x7 'same' window of the 2-channel flow (update.py:92,75: convf1), tap-major then (x, y) channel:
// 98 values per pixel, zero outside the image, as fp16 hi/lo planes of 128 channels (98..127 = 0).
__global__ void flow_im2col_kernel(const float* __restrict__ flow, int B, int h, int w, __half* __restrict__ hi,
                                   __half* __restrict__ lo) {
  const size_t total = (size_t)B * h * w * 128;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int kk = (int)(i & 127);
    const size_t px = i >> 7;
    float v = 0.f;
    if (kk < 98) {
      const int x = (int)(px % w), y = (int)((px / w) % h);
      const int tap = kk >> 1, c = kk & 1;
      const int yy = y + tap / 7 - 3, xx = x + tap % 7 - 3;
      if (yy >= 0 && yy < h && xx >= 0 && xx < w) v = __ldg(flow + (px + (size_t)(yy - y) * w + (xx - x)) * 2 + c);
    }
    __half hh, ll;
    split_f16(v, hh, ll);
    hi[i] = hh;
    lo[i] = ll;
  }
}

// Folded inference BatchNorm: scale = gamma * rsqrt(var + eps), shift = beta - mean * scale.
__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var, float eps, int C,
                               float* __restrict__ scale, float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float s = gamma[c] * rsqrtf(var[c] + eps);
  scale[c] = s;
  shift[c] = beta[c] - mean[c] * s;
}
// tanh / relu split of the context encoder output (model.py:84-86): (npix, hid+ctx) -> net (npix, hid), inp (npix, ctx)
__global__ void context_split_kernel(const float* __restrict__ cnet, size_t npix, int hid, int ctx,
                                     float* __restrict__ net, float* __restrict__ inp) {
  const int C = hid + ctx;
  const size_t total = npix * (size_t)C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t px = i / C;
    const int c = (int)(i - px * C);
    const float v = cnet[i];
    if (c < hid) net[px * hid + c] = tanhf(v);
    else inp[px * ctx + (c - hid)] = fmaxf(v, 0.f);
  }
}

// ------------------------------------------------------------------------------------------------
// Warm start for the next pair of a video (the original RAFT's forward_interpolate): forward-splat
// the flow of one pair and fill every grid point from the nearest splatted sample.
//   Sample i = (x, y) lands at (x + fx, y + fy) (fp64) and is kept iff it lands strictly inside
//   (0, w) x (0, h); NaN never is.  Query q takes the flow of the kept sample with the least
//   d2 = ((qx-x)-fx)^2 + ((qy-y)-fy)^2, every operation an individually rounded fp64 op, ties to the
//   lowest sample index (strict < over samples scanned in index order); no kept sample -> 0.
// Exact brute force, O((h*w)^2) per image: one thread per query, grid (query blocks, B); the block
// stages the image's samples through shared memory in tiles.  A dropped sample is staged with a NaN
// flow, so its d2 is NaN and never compares below the running best.
// ------------------------------------------------------------------------------------------------
constexpr int kFwdInterpThreads = 128;
__global__ void __launch_bounds__(kFwdInterpThreads) forward_interpolate_kernel(const float* __restrict__ flow, int h,
                                                                               int w, int out_coords,
                                                                               float* __restrict__ out) {
  __shared__ double2 s_x[kFwdInterpThreads];           // (x, fx)
  __shared__ double2 s_y[kFwdInterpThreads];           // (y, fy)
  const int n = h * w;
  const float* f = flow + (size_t)blockIdx.y * n * 2;
  const int q = blockIdx.x * kFwdInterpThreads + threadIdx.x;
  const double qx = (double)(q % w), qy = (double)(q / w);
  double best = __longlong_as_double(0x7ff0000000000000ll);   // +inf
  int best_i = -1;
  for (int t0 = 0; t0 < n; t0 += kFwdInterpThreads) {
    const int i = t0 + threadIdx.x;
    if (i < n) {
      const double x = (double)(i % w), y = (double)(i / w);
      const double fx = (double)f[2 * i], fy = (double)f[2 * i + 1];
      const double px = __dadd_rn(x, fx), py = __dadd_rn(y, fy);
      const bool keep = px > 0.0 && px < (double)w && py > 0.0 && py < (double)h;
      s_x[threadIdx.x] = make_double2(x, keep ? fx : __longlong_as_double(0x7ff8000000000000ll));
      s_y[threadIdx.x] = make_double2(y, fy);
    }
    __syncthreads();
    if (q < n) {
      const int m = min(kFwdInterpThreads, n - t0);
#pragma unroll 4
      for (int j = 0; j < m; ++j) {
        const double2 a = s_x[j], b = s_y[j];
        const double dx = __dsub_rn(__dsub_rn(qx, a.x), a.y);
        const double dy = __dsub_rn(__dsub_rn(qy, b.x), b.y);
        const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        if (d2 < best) {
          best = d2;
          best_i = t0 + j;
        }
      }
    }
    __syncthreads();
  }
  if (q >= n) return;
  float vx = 0.0f, vy = 0.0f;
  if (best_i >= 0) {
    vx = f[2 * best_i];
    vy = f[2 * best_i + 1];
  }
  if (out_coords) {                                    // coords_grid + flow: the coords1 the forward loop starts from
    vx = __fadd_rn((float)(q % w), vx);
    vy = __fadd_rn((float)(q / w), vy);
  }
  float* o = out + ((size_t)blockIdx.y * n + q) * 2;
  o[0] = vx;
  o[1] = vy;
}

inline int grid_for(size_t n, int block = 256, int cap = kNumSMs * 16) {
  size_t g = (n + block - 1) / block;
  if (g < 1) g = 1;
  if (g > (size_t)cap) g = cap;
  return (int)g;
}

}  // namespace raft
