// NHWC fp32 implicit-GEMM convolution on the CUDA cores (exact fp32 FMA accumulation, rel. error
// ~1e-6 vs the oracle).  One generic tap-table kernel serves forward convs (3x3 s1, 4x4 s2, 1x1,
// Linear), stride-1 dgrad (tap offsets p-ky) and stride-2 dgrad (four output-parity classes of 2x2
// taps).  It is the exact-precision path: the tcgen05 TF32 kernel (conv_tc.cu) takes the large-M
// layers, this one keeps the skinny-M weight-streaming layers (split-K), the thin layers
// (Cin or Cout == 1) and every weight-gradient GEMM.
//
// Replaces: every nn.Conv2d / nn.ConvTranspose2d / nn.Linear call of arch/Ours/networks.py:18-19,
// 41-46, 170, 181-306 and their autograd backward (ATen convolution_backward).
#include <algorithm>
#include <string.h>
#include <vector>
#include "common.cuh"
#include "mtdgan_b200.h"

namespace {

constexpr int kMaxTaps = 16;

struct ConvArgs {
  const float* src1;
  const float* src2;
  int C1, C2;
  int B, H, W;          // source spatial dims
  const float* wp;      // packed weights [N][T][C1+C2]
  int N, T;
  int Ho, Wo;           // logical output grid of this launch
  int sy, sx;           // source coord = o * s + d[t]
  int dy[kMaxTaps], dx[kMaxTaps];
  float* out;           // (B, outH, outW, N); pixel = (oy*omy+ooy, ox*omx+oox)
  int outH, outW, omy, omx, ooy, oox;
  // epilogue: v = acc*scale + bias; v = pre_act(v); aux = v; v += add1 + add2; v = post_act(v);
  //           v *= act'(mask_src)
  const float* scale;   // device scalar (1/sigma) or null; with scale_span > 0 an array indexed by output element / span
  long long scale_span; // output elements per scale entry (samples per group x outH x outW x N), 0 = one scalar
  const float* bias;
  int pre_act;
  const float* add1;
  const float* add2;
  int post_act;
  const float* mask_src;
  int mask_act;
  float slope;
  float* aux;
  // split-K: when splits > 1 raw partial sums are atomically added into `out` (pre-zeroed) and the
  // epilogue runs in conv_epilogue_kernel.
  int splits;
};

__device__ __forceinline__ float conv_epilogue_one(const ConvArgs& a, float v, size_t idx, int n) {
  if (a.scale) v *= __ldg(a.scale + (a.scale_span > 0 ? (long long)idx / a.scale_span : 0));
  if (a.bias) v += __ldg(a.bias + n);
  v = mtd_act(v, a.pre_act, a.slope);
  if (a.aux) a.aux[idx] = v;
  if (a.add1) v += __ldg(a.add1 + idx);
  if (a.add2) v += __ldg(a.add2 + idx);
  v = mtd_act(v, a.post_act, a.slope);
  if (a.mask_src) v *= mtd_act_grad(__ldg(a.mask_src + idx), a.mask_act, a.slope);
  return v;
}

// four consecutive output channels of one pixel (idx % 4 == 0, N % 4 == 0, 16-byte aligned tensors)
__device__ __forceinline__ float4 conv_epilogue_four(const ConvArgs& a, float4 v, size_t idx, int n) {
  if (a.scale) {
    const float sc = __ldg(a.scale + (a.scale_span > 0 ? (long long)idx / a.scale_span : 0));
    v.x *= sc; v.y *= sc; v.z *= sc; v.w *= sc;
  }
  if (a.bias) { const float4 t = __ldg(reinterpret_cast<const float4*>(a.bias + n)); v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w; }
  v.x = mtd_act(v.x, a.pre_act, a.slope); v.y = mtd_act(v.y, a.pre_act, a.slope);
  v.z = mtd_act(v.z, a.pre_act, a.slope); v.w = mtd_act(v.w, a.pre_act, a.slope);
  if (a.aux) *reinterpret_cast<float4*>(a.aux + idx) = v;
  if (a.add1) { const float4 t = __ldg(reinterpret_cast<const float4*>(a.add1 + idx)); v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w; }
  if (a.add2) { const float4 t = __ldg(reinterpret_cast<const float4*>(a.add2 + idx)); v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w; }
  v.x = mtd_act(v.x, a.post_act, a.slope); v.y = mtd_act(v.y, a.post_act, a.slope);
  v.z = mtd_act(v.z, a.post_act, a.slope); v.w = mtd_act(v.w, a.post_act, a.slope);
  if (a.mask_src) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(a.mask_src + idx));
    v.x *= mtd_act_grad(t.x, a.mask_act, a.slope); v.y *= mtd_act_grad(t.y, a.mask_act, a.slope);
    v.z *= mtd_act_grad(t.z, a.mask_act, a.slope); v.w *= mtd_act_grad(t.w, a.mask_act, a.slope);
  }
  return v;
}

template <int TM, int TN, bool VEC>
__global__ void __launch_bounds__(256) conv_igemm_kernel(const __grid_constant__ ConvArgs a) {
  mtd_pdl_prologue();
  constexpr int BM = 16 * TM, BN = 16 * TN, BK = 16;
  constexpr int A_PER = (BM * 4 + 255) / 256;
  constexpr int B_PER = (BN * 4 + 255) / 256;
  __shared__ __align__(16) float As[2][BK][BM];
  __shared__ __align__(16) float Bs[2][BK][BN];

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int Ctot = a.C1 + a.C2;
  const int HoWo = a.Ho * a.Wo;
  const int M = a.B * HoWo;
  const int nchunk = (Ctot + BK - 1) / BK;
  const int niter = a.T * nchunk;
  int it_begin = 0, it_end = niter;
  if (a.splits > 1) {
    int per = (niter + a.splits - 1) / a.splits;
    it_begin = blockIdx.z * per;
    it_end = min(niter, it_begin + per);
    if (it_begin >= it_end) return;
  }

  // per-slot pixel decode for the A loader (rows are fixed per thread for the whole K loop)
  int a_b[A_PER], a_ys[A_PER], a_xs[A_PER];
  bool a_ok[A_PER];
#pragma unroll
  for (int p = 0; p < A_PER; ++p) {
    int s = tid + p * 256;
    int row = s >> 2;
    int m = m0 + row;
    a_ok[p] = (row < BM) && (m < M);
    int mm = a_ok[p] ? m : 0;
    int b = mm / HoWo, r = mm - b * HoWo;
    int oy = r / a.Wo, ox = r - oy * a.Wo;
    a_b[p] = b;
    a_ys[p] = oy * a.sy;
    a_xs[p] = ox * a.sx;
  }

  float4 ra[A_PER], rb[B_PER];

  auto load_tiles = [&](int it) {
    int t = it / nchunk;
    int c0 = (it - t * nchunk) * BK;
    int ddy = a.dy[t], ddx = a.dx[t];
#pragma unroll
    for (int p = 0; p < A_PER; ++p) {
      int s = tid + p * 256;
      int kq = s & 3;
      int c = c0 + kq * 4;
      int iy = a_ys[p] + ddy, ix = a_xs[p] + ddx;
      bool ok = a_ok[p] && iy >= 0 && iy < a.H && ix >= 0 && ix < a.W;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok) {
        size_t pix = ((size_t)a_b[p] * a.H + iy) * a.W + ix;
        if (VEC) {
          if (c < a.C1) v = __ldg(reinterpret_cast<const float4*>(a.src1 + pix * a.C1 + c));
          else if (c < Ctot) v = __ldg(reinterpret_cast<const float4*>(a.src2 + pix * a.C2 + (c - a.C1)));
        } else {
          float tmp[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            int cc = c + j;
            tmp[j] = cc < a.C1 ? __ldg(a.src1 + pix * a.C1 + cc)
                               : (cc < Ctot ? __ldg(a.src2 + pix * a.C2 + (cc - a.C1)) : 0.f);
          }
          v = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
        }
      }
      ra[p] = v;
    }
#pragma unroll
    for (int p = 0; p < B_PER; ++p) {
      int s = tid + p * 256;
      int row = s >> 2, kq = s & 3;
      int n = n0 + row;
      int c = c0 + kq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < BN && n < a.N) {
        const float* wrow = a.wp + ((size_t)n * a.T + t) * Ctot;
        if (VEC) {
          if (c < Ctot) v = __ldg(reinterpret_cast<const float4*>(wrow + c));
        } else {
          float tmp[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) tmp[j] = (c + j < Ctot) ? __ldg(wrow + c + j) : 0.f;
          v = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
        }
      }
      rb[p] = v;
    }
  };

  auto store_tiles = [&](int buf) {
#pragma unroll
    for (int p = 0; p < A_PER; ++p) {
      int s = tid + p * 256;
      int row = s >> 2, kq = s & 3;
      if (row < BM) {
        As[buf][kq * 4 + 0][row] = ra[p].x;
        As[buf][kq * 4 + 1][row] = ra[p].y;
        As[buf][kq * 4 + 2][row] = ra[p].z;
        As[buf][kq * 4 + 3][row] = ra[p].w;
      }
    }
#pragma unroll
    for (int p = 0; p < B_PER; ++p) {
      int s = tid + p * 256;
      int row = s >> 2, kq = s & 3;
      if (row < BN) {
        Bs[buf][kq * 4 + 0][row] = rb[p].x;
        Bs[buf][kq * 4 + 1][row] = rb[p].y;
        Bs[buf][kq * 4 + 2][row] = rb[p].z;
        Bs[buf][kq * 4 + 3][row] = rb[p].w;
      }
    }
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  load_tiles(it_begin);
  store_tiles(0);
  __syncthreads();
  int buf = 0;
  for (int it = it_begin; it < it_end; ++it) {
    bool has_next = (it + 1) < it_end;
    if (has_next) load_tiles(it + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float av[TM], bv[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) av[i] = As[buf][k][ty * TM + i];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[buf][k][tx * TN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (has_next) store_tiles(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }

  // epilogue
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int m = m0 + ty * TM + i;
    if (m >= M) continue;
    int b = m / HoWo, r = m - b * HoWo;
    int oy = r / a.Wo, ox = r - oy * a.Wo;
    size_t pix = ((size_t)b * a.outH + (oy * a.omy + a.ooy)) * a.outW + (ox * a.omx + a.oox);
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int n = n0 + tx * TN + j;
      if (n >= a.N) continue;
      size_t idx = pix * a.N + n;
      if (a.splits > 1) atomicAdd(a.out + idx, acc[i][j]);
      else a.out[idx] = conv_epilogue_one(a, acc[i][j], idx, n);
    }
  }
}


// ---------------------------------------------------------------------------------------------------
// Thin layers (bandwidth-bound, no GEMM shape): dedicated streaming kernels instead of padded tiles.
//   conv_c1_kernel : source has ONE channel   out[p][n] = epi( sum_t in[p@t] * W[n][t] )
//                    (conv11 1->64, generator encoder[0] 1->32, the 1->1 heads; dgrad of every Cout = 1 layer)
//   conv_n1_kernel : N <= 4 outputs            out[p][n] = epi( sum_t sum_c in[p@t][c] * W[n][t][c] )
//                    (s_/r_dconv61 128->1, generator decoder[0] 32->1; dgrad of every Cin = 1 layer)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv_c1_kernel(const __grid_constant__ ConvArgs a, int vec4) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) float wsm[];   // [T][N4]  (N padded to a multiple of 4, zero filled)
  const int N4 = (a.N + 3) & ~3;
  for (int i = threadIdx.x; i < a.T * N4; i += blockDim.x) {
    int t = i / N4, n = i - t * N4;
    wsm[i] = n < a.N ? __ldg(a.wp + (size_t)n * a.T + t) : 0.f;
  }
  __syncthreads();
  const int NQ = N4 >> 2;
  const int HoWo = a.Ho * a.Wo;
  const unsigned total = (unsigned)a.B * HoWo * NQ;            // < 2^32 (checked by the launcher): 32-bit index arithmetic
  unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned stride = gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int nq = (int)(i % (unsigned)NQ);
    const unsigned m = i / (unsigned)NQ;
    const int b = (int)(m / (unsigned)HoWo), r = (int)(m - (unsigned)b * HoWo);
    const int oy = r / a.Wo, ox = r - oy * a.Wo;
    const float* img = a.src1 + (size_t)b * a.H * a.W;
    float v[kMaxTaps];
#pragma unroll
    for (int t = 0; t < kMaxTaps; ++t) {           // all taps' loads in flight together
      v[t] = 0.f;
      if (t < a.T) {
        const int iy = oy * a.sy + a.dy[t], ix = ox * a.sx + a.dx[t];
        if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W) v[t] = __ldg(img + (size_t)iy * a.W + ix);
      }
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int t = 0; t < kMaxTaps; ++t) {
      if (t < a.T) {
        const float4 w = *reinterpret_cast<const float4*>(wsm + t * N4 + nq * 4);
        acc.x = fmaf(v[t], w.x, acc.x); acc.y = fmaf(v[t], w.y, acc.y);
        acc.z = fmaf(v[t], w.z, acc.z); acc.w = fmaf(v[t], w.w, acc.w);
      }
    }
    const size_t pix = ((size_t)b * a.outH + (oy * a.omy + a.ooy)) * a.outW + (ox * a.omx + a.oox);
    if (vec4) {                                     // N % 4 == 0 and 16-byte aligned epilogue operands: one 16-byte store
      const size_t idx = pix * a.N + nq * 4;
      *reinterpret_cast<float4*>(a.out + idx) = conv_epilogue_four(a, acc, idx, nq * 4);
      continue;
    }
    const float accv[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int n = nq * 4 + e;
      if (n < a.N) {
        const size_t idx = pix * a.N + n;
        a.out[idx] = conv_epilogue_one(a, accv[e], idx, n);
      }
    }
  }
}

// LPP lanes cooperate on one pixel (LPP = min(32, Ctot/4)); N <= 4 accumulators per lane, shuffle-reduced.
// Requires Ctot == 4 * LPP * k; the generic case loops over channel groups.
__global__ void __launch_bounds__(256) conv_n1_kernel(const __grid_constant__ ConvArgs a, int lpp) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) float wsm[];   // [N][T][Ctot]
  const int Ctot = a.C1 + a.C2;
  for (int i = threadIdx.x; i < a.N * a.T * Ctot; i += blockDim.x) wsm[i] = __ldg(a.wp + i);
  __syncthreads();
  const int HoWo = a.Ho * a.Wo;
  const size_t M = (size_t)a.B * HoWo;
  const int ppw = 32 / lpp;                       // pixels per warp
  const int lane = threadIdx.x & 31, sub = lane / lpp, l = lane - sub * lpp;
  const size_t warp_global = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t m0 = warp_global * ppw; m0 < M; m0 += nwarps * ppw) {
    const size_t m = m0 + sub;
    const bool valid = m < M;
    const size_t mm = valid ? m : 0;
    const int b = (int)(mm / HoWo), r = (int)(mm - (size_t)b * HoWo);
    const int oy = r / a.Wo, ox = r - oy * a.Wo;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = l * 4; c < Ctot; c += lpp * 4) {
      const float* src = c < a.C1 ? a.src1 + c : a.src2 + (c - a.C1);
      const int Cs = c < a.C1 ? a.C1 : a.C2;
      float4 v[kMaxTaps];
#pragma unroll
      for (int t = 0; t < kMaxTaps; ++t) {         // all taps' loads in flight together
        v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < a.T && valid) {
          const int iy = oy * a.sy + a.dy[t], ix = ox * a.sx + a.dx[t];
          if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W)
            v[t] = __ldg(reinterpret_cast<const float4*>(src + (((size_t)b * a.H + iy) * a.W + ix) * Cs));
        }
      }
#pragma unroll
      for (int t = 0; t < kMaxTaps; ++t) {
        if (t < a.T) {
#pragma unroll
          for (int n = 0; n < 4; ++n) {
            if (n < a.N) {
              const float4 w = *reinterpret_cast<const float4*>(wsm + ((size_t)n * a.T + t) * Ctot + c);
              acc[n] = fmaf(v[t].x, w.x, fmaf(v[t].y, w.y, fmaf(v[t].z, w.z, fmaf(v[t].w, w.w, acc[n]))));
            }
          }
        }
      }
    }
#pragma unroll
    for (int n = 0; n < 4; ++n)
      for (int o = lpp >> 1; o > 0; o >>= 1) acc[n] += __shfl_xor_sync(0xffffffffu, acc[n], o);
    if (valid && l == 0) {
      const size_t pix = ((size_t)b * a.outH + (oy * a.omy + a.ooy)) * a.outW + (ox * a.omx + a.oox);
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        if (n < a.N) {
          const size_t idx = pix * a.N + n;
          a.out[idx] = conv_epilogue_one(a, acc[n], idx, n);
        }
      }
    }
  }
}

// N = 1 output channel, 3 x 3 taps, stride 1 (s_dconv61 / r_dconv61 128 -> 1, generator decoder[0] 32 -> 1, data gradient of
// the 1 -> 64 stem): tile version.  out[p] = sum_t in[p + d_t] . w[t] = sum_t q_t[p + d_t] with q_t[p'] = in[p'] . w[t]:
// every input pixel of an (8+2) x (64+2) halo tile is read ONCE (float4 per lane, Ctot/4 lanes per pixel, the lane's 36
// weights in registers), its nine per-tap dot products go to shared memory, then each output pixel gathers nine scalars.
// The pixel-major kernel above re-reads every input pixel nine times through L1/L2 (130 us for 84 MB at B = 40).
constexpr int kN1TileH = 8, kN1TileW = 64, kN1HaloW = kN1TileW + 2, kN1HaloPix = (kN1TileH + 2) * kN1HaloW;

// One THREAD per halo pixel: its Ctot channels are consecutive in memory (NHWC), read as float4s with several loads in
// flight; the nine tap weights of a channel quad come from shared memory as warp-wide broadcasts.  No cross-lane
// reduction: the nine dot products of a pixel live in nine registers of its thread.
__global__ void __launch_bounds__(256) conv_n1t_kernel(const __grid_constant__ ConvArgs a) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) float n1_smem[];
  const int Ctot = a.C1 + a.C2, C4 = Ctot >> 2;
  float4* w4 = reinterpret_cast<float4*>(n1_smem);                  // [9][Ctot/4]
  float* q = n1_smem + 9 * Ctot;                                    // [halo pixel][9]
  for (int i = threadIdx.x; i < 9 * C4; i += blockDim.x) w4[i] = __ldg(reinterpret_cast<const float4*>(a.wp) + i);
  const int tiles_x = a.W / kN1TileW, tiles_y = a.H / kN1TileH;
  int tile = blockIdx.x;
  const int tx = tile % tiles_x; tile /= tiles_x;
  const int ty = tile % tiles_y;
  const int b = tile / tiles_y;
  const int y0 = ty * kN1TileH - 1, x0 = tx * kN1TileW - 1;
  __syncthreads();
  for (int hp = threadIdx.x; hp < kN1HaloPix; hp += blockDim.x) {
    const int hy = hp / kN1HaloW, hx = hp - hy * kN1HaloW;
    const int y = y0 + hy, x = x0 + hx;
    float s[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) s[t] = 0.f;
    if (y >= 0 && y < a.H && x >= 0 && x < a.W) {
      const size_t pix = ((size_t)b * a.H + y) * a.W + x;
      for (int src = 0; src < 2; ++src) {
        const int Cs = src == 0 ? a.C1 : a.C2;
        if (Cs == 0) continue;
        const float4* p = reinterpret_cast<const float4*>((src == 0 ? a.src1 : a.src2) + pix * Cs);
        const float4* wq = w4 + (src == 0 ? 0 : (a.C1 >> 2));
        for (int c0 = 0; c0 < (Cs >> 2); c0 += 4) {          // Cs is a multiple of 16 (32 / 64 / 128 channel layers)
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) v[u] = __ldg(p + c0 + u);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int t = 0; t < 9; ++t) {
              const float4 w = wq[t * C4 + c0 + u];
              s[t] = fmaf(v[u].x, w.x, fmaf(v[u].y, w.y, fmaf(v[u].z, w.z, fmaf(v[u].w, w.w, s[t]))));
            }
          }
        }
      }
    }
#pragma unroll
    for (int t = 0; t < 9; ++t) q[hp * 9 + t] = s[t];
  }
  __syncthreads();
  for (int op = threadIdx.x; op < kN1TileH * kN1TileW; op += blockDim.x) {
    const int oy = op / kN1TileW, ox = op - oy * kN1TileW;
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) acc += q[((oy + 1 + a.dy[t]) * kN1HaloW + (ox + 1 + a.dx[t])) * 9 + t];
    const size_t idx = ((size_t)b * a.H + (ty * kN1TileH + oy)) * a.W + (tx * kN1TileW + ox);
    a.out[idx] = conv_epilogue_one(a, acc, idx, 0);
  }
}

// Thin weight gradient: out[t*st_t + j*st_j] += sum_p V[p][j] * s[p + d_t]  (s: single-channel field of the same
// spatial size as V's pixel grid, zero outside).  Covers wgrad of Cout = 1 layers (s = dz, V = x, d_t = -tap) and of
// Cin = 1 layers (s = x, V = dz, d_t = +tap).  L = J/4 lanes cover one pixel's J channels with float4 loads (32/L
// pixels per warp per iteration); block-level reduction in shared memory, one atomicAdd per (t, j) per block.
struct ThinWgArgs {
  const float* V1;
  const float* V2;
  int J1, J2;              // vector channels per source
  const float* s;
  int B, H, W, T;
  int dy[kMaxTaps], dx[kMaxTaps];
  float* out;
  long long st_t, st_j;
  int pix_per_block;
};

template <bool VEC4>
__global__ void __launch_bounds__(256) thin_wgrad_kernel(const __grid_constant__ ThinWgArgs a) {
  mtd_pdl_prologue();
  extern __shared__ float red[];                        // [T][J]
  const int J = a.J1 + a.J2;
  const int HW = a.H * a.W;
  const long long M = (long long)a.B * HW;
  const long long p0 = (long long)blockIdx.x * a.pix_per_block;
  const long long p1 = min(M, p0 + a.pix_per_block);
  for (int i = threadIdx.x; i < a.T * J; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  constexpr int E = VEC4 ? 4 : 1;
  const int L = VEC4 ? (J >> 2) : J;                    // threads per pixel
  const int pl = threadIdx.x / L, jl = threadIdx.x - pl * L, npl = blockDim.x / L;
  float acc[kMaxTaps][E];
#pragma unroll
  for (int t = 0; t < kMaxTaps; ++t)
#pragma unroll
    for (int e = 0; e < E; ++e) acc[t][e] = 0.f;
  if (pl < npl) {
    const int j = jl * E;
    for (long long p = p0 + pl; p < p1; p += npl) {
      float v[E];
      if (VEC4) {
        const float4 t4 = j < a.J1 ? __ldg(reinterpret_cast<const float4*>(a.V1 + p * a.J1 + j))
                                   : __ldg(reinterpret_cast<const float4*>(a.V2 + p * a.J2 + (j - a.J1)));
        v[0] = t4.x; if (E > 1) { v[E > 1 ? 1 : 0] = t4.y; v[E > 2 ? 2 : 0] = t4.z; v[E > 3 ? 3 : 0] = t4.w; }
      } else {
        v[0] = j < a.J1 ? __ldg(a.V1 + p * a.J1 + j) : __ldg(a.V2 + p * a.J2 + (j - a.J1));
      }
      const int b = (int)(p / HW), r = (int)(p - (long long)b * HW);
      const int y = r / a.W, x = r - y * a.W;
      float sv[kMaxTaps];
#pragma unroll
      for (int t = 0; t < kMaxTaps; ++t) {
        sv[t] = 0.f;
        if (t < a.T) {
          const int yy = y + a.dy[t], xx = x + a.dx[t];
          if (yy >= 0 && yy < a.H && xx >= 0 && xx < a.W) sv[t] = __ldg(a.s + ((size_t)b * a.H + yy) * a.W + xx);
        }
      }
#pragma unroll
      for (int t = 0; t < kMaxTaps; ++t)
#pragma unroll
        for (int e = 0; e < E; ++e) acc[t][e] = fmaf(v[e], sv[t], acc[t][e]);
    }
    for (int t = 0; t < a.T; ++t)
#pragma unroll
      for (int e = 0; e < E; ++e) atomicAdd(&red[t * J + j + e], acc[t][e]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < a.T * J; i += blockDim.x) {
    const int t = i / J, j = i - t * J;
    atomicAdd(a.out + t * a.st_t + j * a.st_j, red[i]);
  }
}

// second phase of a split-K conv: out holds raw sums
__global__ void conv_epilogue_kernel(const __grid_constant__ ConvArgs a, size_t total) {
  mtd_pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int n = (int)(i % a.N);
    a.out[i] = conv_epilogue_one(a, a.out[i], i, n);
  }
}

// conv_c1 with 16 output channels per thread (N % 16 == 0, vector epilogue): the nine source loads and their bounds
// arithmetic are shared by four float4 groups instead of being repeated by each of them.
__global__ void __launch_bounds__(256) conv_c1x16_kernel(const __grid_constant__ ConvArgs a) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) float wsm[];   // [T][N]
  for (int i = threadIdx.x; i < a.T * a.N; i += blockDim.x) {
    int t = i / a.N, n = i - t * a.N;
    wsm[i] = __ldg(a.wp + (size_t)n * a.T + t);
  }
  __syncthreads();
  const int NG = a.N >> 4;
  const int HoWo = a.Ho * a.Wo;
  const unsigned total = (unsigned)a.B * HoWo * NG;
  unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned stride = gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int ng = (int)(i % (unsigned)NG);
    const unsigned m = i / (unsigned)NG;
    const int b = (int)(m / (unsigned)HoWo), r = (int)(m - (unsigned)b * HoWo);
    const int oy = r / a.Wo, ox = r - oy * a.Wo;
    const float* img = a.src1 + (size_t)b * a.H * a.W;
    float v[kMaxTaps];
#pragma unroll
    for (int t = 0; t < kMaxTaps; ++t) {
      v[t] = 0.f;
      if (t < a.T) {
        const int iy = oy * a.sy + a.dy[t], ix = ox * a.sx + a.dx[t];
        if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W) v[t] = __ldg(img + (size_t)iy * a.W + ix);
      }
    }
    float4 acc[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int t = 0; t < kMaxTaps; ++t) {
      if (t < a.T) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 w = *reinterpret_cast<const float4*>(wsm + t * a.N + ng * 16 + q * 4);
          acc[q].x = fmaf(v[t], w.x, acc[q].x); acc[q].y = fmaf(v[t], w.y, acc[q].y);
          acc[q].z = fmaf(v[t], w.z, acc[q].z); acc[q].w = fmaf(v[t], w.w, acc[q].w);
        }
      }
    }
    const size_t pix = ((size_t)b * a.outH + (oy * a.omy + a.ooy)) * a.outW + (ox * a.omx + a.oox);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int n = ng * 16 + q * 4;
      const size_t idx = pix * a.N + n;
      *reinterpret_cast<float4*>(a.out + idx) = conv_epilogue_four(a, acc[q], idx, n);
    }
  }
}

int launch_conv(ConvArgs& a, cudaStream_t st) {
  const int Ctot = a.C1 + a.C2;
  const int M = a.B * a.Ho * a.Wo;
  if (M <= 0 || a.N <= 0 || Ctot <= 0 || a.T <= 0 || a.T > kMaxTaps) return MTD_EINVAL;
  bool vec = (a.C1 % 4 == 0) && (a.C2 % 4 == 0) && mtd_aligned16(a.src1) && mtd_aligned16(a.wp) &&
             (a.C2 == 0 || mtd_aligned16(a.src2));
  a.splits = 1;
  if (Ctot == 1 && a.T * a.N * sizeof(float) <= 40 * 1024 && (size_t)M * ((a.N + 3) / 4) < (1ull << 31)) {   // single-channel source
    size_t work = (size_t)M * ((a.N + 3) / 4);
    int blocks = (int)std::min<size_t>((work + 255) / 256, (size_t)mtd_sm_count() * 16);
    auto al = [](const void* p) { return p == nullptr || mtd_aligned16(p); };
    const int vec4 = (a.N % 4 == 0 && mtd_aligned16(a.out) && al(a.bias) && al(a.add1) && al(a.add2) && al(a.mask_src) && al(a.aux) &&
                      (a.scale_span == 0 || a.scale_span % 4 == 0)) ? 1 : 0;
    if (vec4 && a.N % 16 == 0 && (size_t)M * (a.N / 16) >= (size_t)mtd_sm_count() * 256 * 4) {
      work = (size_t)M * (a.N / 16);
      blocks = (int)std::min<size_t>((work + 255) / 256, (size_t)mtd_sm_count() * 16);
      mtd_launch(conv_c1x16_kernel, blocks, 256, a.T * a.N * sizeof(float), st, a);
    } else {
      mtd_launch(conv_c1_kernel, blocks, 256, a.T * ((a.N + 3) & ~3) * sizeof(float), st, a, vec4);
    }
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
  {   // N = 1, 3 x 3 neighbourhood, stride 1, dense output: halo-tile kernel (every input pixel read once)
    bool nb = a.N == 1 && a.T == 9 && a.sy == 1 && a.sx == 1 && a.Ho == a.H && a.Wo == a.W && a.outH == a.H && a.outW == a.W &&
              a.omy == 1 && a.omx == 1 && a.ooy == 0 && a.oox == 0 && vec && a.C1 % 16 == 0 && a.C2 % 16 == 0 && Ctot <= 256 &&
              a.W % kN1TileW == 0 && a.H % kN1TileH == 0;
    for (int t = 0; nb && t < 9; ++t) nb = a.dy[t] >= -1 && a.dy[t] <= 1 && a.dx[t] >= -1 && a.dx[t] <= 1;
    if (nb) {
      const int tiles = a.B * (a.H / kN1TileH) * (a.W / kN1TileW);
      mtd_launch(conv_n1t_kernel, tiles, 256, (size_t)(9 * Ctot + kN1HaloPix * 9) * sizeof(float), st, a);
      MTD_CHECK_LAUNCH();
      return MTD_OK;
    }
  }
  if (a.N <= 4 && vec && Ctot >= 8 && (size_t)a.N * a.T * Ctot * sizeof(float) <= 40 * 1024) {   // few outputs, many channels
    int lpp = 1;
    while (lpp < 32 && lpp * 2 * 4 <= Ctot) lpp <<= 1;
    size_t warps = ((size_t)M + (32 / lpp) - 1) / (32 / lpp);
    int blocks = (int)std::min<size_t>((warps + 7) / 8, (size_t)mtd_sm_count() * 16);
    mtd_launch(conv_n1_kernel, blocks, 256, (size_t)a.N * a.T * Ctot * sizeof(float), st, a, lpp);
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
  bool thin_n = a.N <= 16;
  const int BM = thin_n ? 128 : 64, BN = thin_n ? 16 : 64;
  dim3 grid((M + BM - 1) / BM, (a.N + BN - 1) / BN, 1);
  const int niter = a.T * ((Ctot + 15) / 16);
  int ctas = grid.x * grid.y;
  int splits = 1;
  const int target = 2 * mtd_sm_count();
  bool full_out = (a.omy == 1 && a.omx == 1);   // split-K epilogue pass assumes a dense output
  if (ctas < target && niter >= 16 && full_out) {
    splits = std::min((target + ctas - 1) / ctas, niter / 8);
    if (splits < 1) splits = 1;
    if (splits > 64) splits = 64;
  }
  a.splits = splits;
  grid.z = splits;
  size_t total = (size_t)a.B * a.outH * a.outW * a.N;
  if (splits > 1) MTD_CUDA(cudaMemsetAsync(a.out, 0, total * sizeof(float), st));
  if (thin_n) {
    if (vec) mtd_launch(conv_igemm_kernel<8, 1, true>, grid, 256, 0, st, a);
    else mtd_launch(conv_igemm_kernel<8, 1, false>, grid, 256, 0, st, a);
  } else {
    if (vec) mtd_launch(conv_igemm_kernel<4, 4, true>, grid, 256, 0, st, a);
    else mtd_launch(conv_igemm_kernel<4, 4, false>, grid, 256, 0, st, a);
  }
  MTD_CHECK_LAUNCH();
  if (splits > 1) {
    int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)mtd_sm_count() * 8);
    mtd_launch(conv_epilogue_kernel, blocks, 256, 0, st, a, total);
    MTD_CHECK_LAUNCH();
  }
  return MTD_OK;
}

// ---------------------------------------------------------------------------------------------
// weight packing:  out[n][t][c] = w[n*sN + c*sC + toff[t]]   (and its inverse for gradients)
// ---------------------------------------------------------------------------------------------
struct PackArgs {
  int N, T, C;
  long long sN, sC;
  int toff[kMaxTaps];
  int blocked;     // 1: tile-major layout [N/32][T*C/32][32 n][32 k] (every 32x32 tile = 4 KB contiguous) for the TMA /
                   //    tcgen05 kernels: a weight tile is a few contiguous 4 KB runs instead of 128 B pieces 4*T*C bytes apart
  int tf32;        // 0: fp32 copy; 1: rounded to tf32 (nearest); 3: tf32 hi at out[o], tf32 residual at out[o + lo_off]
  long long lo_off;
};

__global__ void pack_weights_kernel(const float* __restrict__ w, float* __restrict__ out, const __grid_constant__ PackArgs p) {
  mtd_pdl_prologue();
  size_t total = (size_t)p.N * p.T * p.C;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int c = (int)(i % p.C);
    size_t r = i / p.C;
    int t = (int)(r % p.T);
    int n = (int)(r / p.T);
    size_t o = i;
    if (p.blocked) {
      const size_t k = (size_t)t * p.C + c, KS = (size_t)p.T * p.C / 32;
      o = ((((size_t)(n >> 5) * KS + (k >> 5)) * 32 + (n & 31)) << 5) + (k & 31);
    }
    const float v = __ldg(w + (size_t)n * p.sN + (size_t)c * p.sC + p.toff[t]);
    if (p.tf32 == 0) { out[o] = v; continue; }
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
    out[o] = __uint_as_float(h);
    if (p.tf32 == 3) {
      uint32_t l;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - __uint_as_float(h)));     // the residual is exact in fp32
      out[o + p.lo_off] = __uint_as_float(l);
    }
  }
}

// Batched packing: up to kPackBatch packs per launch, described in kernel-parameter space (no table upload), so the
// ~230 per-layer pack launches of a train step (every weight changes once per step) become ~10.
constexpr int kPackBatch = 24;
constexpr int kPackChunk = 8192;          // elements per block
struct PackBatch {
  const float* w[kPackBatch];
  float* out[kPackBatch];
  PackArgs p[kPackBatch];
  int first_block[kPackBatch + 1];        // prefix sums of blocks per pack
  int n;
};
static_assert(sizeof(PackBatch) <= 4000, "PackBatch must fit the kernel parameter space");

__device__ __forceinline__ void pack_one(const float* __restrict__ w, float* __restrict__ out, const PackArgs& p, size_t i) {
  int c = (int)(i % p.C);
  size_t r = i / p.C;
  int t = (int)(r % p.T);
  int n = (int)(r / p.T);
  size_t o = i;
  if (p.blocked) {
    const size_t k = (size_t)t * p.C + c, KS = (size_t)p.T * p.C / 32;
    o = ((((size_t)(n >> 5) * KS + (k >> 5)) * 32 + (n & 31)) << 5) + (k & 31);
  }
  const float v = __ldg(w + (size_t)n * p.sN + (size_t)c * p.sC + p.toff[t]);
  if (p.tf32 == 0) { out[o] = v; return; }
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
  out[o] = __uint_as_float(h);
  if (p.tf32 == 3) {
    uint32_t l;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - __uint_as_float(h)));
    out[o + p.lo_off] = __uint_as_float(l);
  }
}

__global__ void __launch_bounds__(256) pack_batched_kernel(const __grid_constant__ PackBatch pb) {
  mtd_pdl_prologue();
  int s = 0;
  while (s + 1 < pb.n && (int)blockIdx.x >= pb.first_block[s + 1]) ++s;
  const PackArgs& p = pb.p[s];
  const size_t total = (size_t)p.N * p.T * p.C;
  const size_t begin = (size_t)((int)blockIdx.x - pb.first_block[s]) * kPackChunk;
  const size_t end = min(total, begin + (size_t)kPackChunk);
  for (size_t i = begin + threadIdx.x; i < end; i += blockDim.x) pack_one(pb.w[s], pb.out[s], p, i);
}

// dw_ref[n*sN + c*sC + toff[t]] = alpha * (gp[n][t][c] - beta * u[n_sn] * v[k_sn])
// where for spectral-normed layers alpha = 1/sigma, beta = <G,W>/sigma and (u,v) index the
// (Cout, Cin*kh*kw) matrix view of the REFERENCE layout (SURVEY A5).
struct UnpackArgs {
  PackArgs p;
  const float* inv_sigma;   // null => plain layer
  const double* dotgw;      // device scalar <G, W_orig> (fp64 accumulator of dot_packed_ref_kernel)
  const float* u;
  const float* v;
  int sn_rows;              // Cout of the reference weight; row = ref_index / sn_cols
  long long sn_cols;
};

__global__ void unpack_grad_kernel(const float* __restrict__ gp, float* __restrict__ dw, const __grid_constant__ UnpackArgs a) {
  mtd_pdl_prologue();
  const PackArgs& p = a.p;
  size_t total = (size_t)p.N * p.T * p.C;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  float alpha = 1.f, beta = 0.f;
  if (a.inv_sigma) {
    alpha = __ldg(a.inv_sigma);
    beta = (float)(*a.dotgw) * alpha;
  }
  for (; i < total; i += stride) {
    int c = (int)(i % p.C);
    size_t r = i / p.C;
    int t = (int)(r % p.T);
    int n = (int)(r / p.T);
    size_t ref = (size_t)n * p.sN + (size_t)c * p.sC + p.toff[t];
    float g = gp[i];
    if (a.inv_sigma) {
      size_t row = ref / a.sn_cols, col = ref - row * a.sn_cols;
      g = alpha * (g - beta * __ldg(a.u + row) * __ldg(a.v + col));
    }
    dw[ref] = g;
  }
}

// <gp, w_ref> with the same index mapping; fp64 accumulation, one atomicAdd(double) per block,
// final value converted by dot_finish_kernel.
__global__ void dot_packed_ref_kernel(const float* __restrict__ gp, const float* __restrict__ w, double* __restrict__ acc,
                                      const __grid_constant__ PackArgs p) {
  mtd_pdl_prologue();
  __shared__ double sh[32];
  size_t total = (size_t)p.N * p.T * p.C;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  double s = 0.0;
  for (; i < total; i += stride) {
    int c = (int)(i % p.C);
    size_t r = i / p.C;
    int t = (int)(r % p.T);
    int n = (int)(r / p.T);
    s += (double)gp[i] * (double)__ldg(w + (size_t)n * p.sN + (size_t)c * p.sC + p.toff[t]);
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) atomicAdd(acc, s);
}


// ---------------------------------------------------------------------------------------------------
// Batched weight-gradient finishing: ONE dot launch + ONE unpack launch for all layers of a backward pass
// (instead of two launches per layer), which also SUMS the contributions of the several forward instances that
// used the same weight (the discriminator runs 2-4 times inside one d_loss graph) — replacing autograd's
// per-instance add kernels.  Segment = one (layer, forward instance), 16 x int64: { gp, dw, w_ref, u, v, inv_sigma,
// N, T, C, sN, sC, flip, sn_cols, dot slot index, next segment of the same weight (-1 = last), 0 };
// chunk tables (int32[nchunk][2]) = { segment, element offset }: all segments for the dot pass, list heads only
// for the unpack pass.
// ---------------------------------------------------------------------------------------------------
constexpr int kFinChunk = 9216;        // >= the longest packed row of the model (3*3*1024, 4*4*512)
struct FinSeg {
  const float* gp;
  float* dw;
  const float* w;
  const float* u;
  const float* v;
  const float* inv_sigma;
  long long N, T, C, sN, sC, flip, sn_cols, slot, next;
  const double* dot_zw;     // optional: sum over this instance's pixels of dz . (W (*) x), computed by mtd_act_bwd_sn (then no dot pass)
};
static_assert(sizeof(FinSeg) == 128, "finish segment must be 16 x int64");

__device__ __forceinline__ size_t fin_ref_index(const FinSeg& s, size_t i) {
  const int c = (int)(i % s.C);
  const size_t r = i / s.C;
  const int t = (int)(r % s.T);
  const size_t n = r / s.T;
  const long long toff = (s.flip & 1) ? (s.T - 1 - t) : t;
  return n * (size_t)s.sN + (size_t)c * s.sC + toff;
}

// A chunk is a whole number of packed rows n (T*C elements each) whenever a row fits (fin_chunk_elems), so for the
// Conv2d / Linear layout its reference-layout image is ONE contiguous range and the (t,c) -> (c,t) permutation can go
// through shared memory: global reads and writes are both coalesced (the element-wise version wrote 4-byte words
// 36 bytes apart and ran at ~1/15 of HBM bandwidth on the 240 MB of discriminator gradients per PCGrad task).
__host__ __device__ inline long long fin_chunk_elems(long long T, long long C) {
  const long long row = T * C;
  return row <= kFinChunk ? (kFinChunk / row) * row : kFinChunk;
}
constexpr long long kFinFlip = 1, kFinPrescaled = 2, kFinNoGp = 4;     // bits of FinSeg::flip
__device__ __forceinline__ bool fin_row_major(const FinSeg& s) {
  return !(s.flip & kFinFlip) && s.sC == s.T && s.sN == s.T * s.C && s.T * s.C <= kFinChunk;
}
__device__ __forceinline__ int fin_pad(int i) { return i + (i >> 5); }      // keeps stride-T (T = 16) accesses conflict-free
constexpr int kFinSmem = kFinChunk + kFinChunk / 32 + 1;

__global__ void __launch_bounds__(256) finish_dot_kernel(const FinSeg* __restrict__ segs, const int2* __restrict__ chunks,
                                                         double* __restrict__ dots) {
  mtd_pdl_prologue();
  __shared__ double sh[32];
  __shared__ float sm[kFinSmem];
  const int2 ck = chunks[blockIdx.x];
  const FinSeg s = segs[ck.x];
  if (!s.inv_sigma) return;                         // uniform per block
  const size_t total = (size_t)s.N * s.T * s.C;
  const size_t end = min(total, (size_t)ck.y + (size_t)fin_chunk_elems(s.T, s.C));
  double acc = 0.0;
  if (fin_row_major(s)) {
    const int cnt = (int)(end - ck.y), T = (int)s.T, C = (int)s.C, row = T * C;
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) sm[fin_pad(j)] = __ldg(s.w + ck.y + j);   // reference order
    __syncthreads();
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) {                                         // packed order
      const int c = j % C, r = j / C, t = r % T, nl = r / T;
      acc += (double)s.gp[ck.y + j] * (double)sm[fin_pad(nl * row + c * T + t)];
    }
  } else {
    for (size_t i = (size_t)ck.y + threadIdx.x; i < end; i += blockDim.x)
      acc += (double)s.gp[i] * (double)__ldg(s.w + fin_ref_index(s, i));
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) atomicAdd(dots + s.slot, acc);
}

// Accumulate, for one chunk of whole packed rows, every forward instance of the weight into shared memory at the
// reference-layout position.  TT > 0: compile-time tap count; CPOW2: channel count is a power of two.
template <int TT, bool CPOW2>
__device__ __forceinline__ void fin_accumulate(const FinSeg* __restrict__ segs, int2 ck, const double* __restrict__ dots, float* sm,
                                               int cnt, int C, int n0) {
  const int T = TT > 0 ? TT : (int)segs[ck.x].T;
  const int row = T * C;
  const int lc = CPOW2 ? (__ffs(C) - 1) : 0;
  long long si = ck.x;
  while (si >= 0) {                                   // every forward instance (and batched group) that used this weight
    const FinSeg& s = segs[si];
    const float* gp = s.gp + ck.y;
    if (s.inv_sigma) {
      const float alpha = __ldg(s.inv_sigma);
      // <G, W~> = <G, W_orig> / sigma; from the activations it is alpha^-1 * sum dz.(y_pre - b) * alpha = that sum itself
      const float beta = s.dot_zw ? (float)(*s.dot_zw) : (float)dots[s.slot] * alpha;
      const float coef = alpha * beta;                // dW = a_gp * gp - coef * u v^T
      const bool nogp = (s.flip & kFinNoGp) != 0;     // correction-only instance (its gp is part of another instance's)
      const float a_gp = (s.flip & kFinPrescaled) ? 1.f : alpha;
      for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
        const int c = CPOW2 ? (j & (C - 1)) : (j % C), r = CPOW2 ? (j >> lc) : (j / C);
        const int nl = r / T, t = r - nl * T;
        const int col = c * T + t;                    // reference (Cout, Cin*kh*kw) matrix view: row = n, col = c*T + t
        const float g = (nogp ? 0.f : a_gp * gp[j]) - coef * __ldg(s.u + n0 + nl) * __ldg(s.v + col);
        sm[fin_pad(nl * row + col)] += g;
      }
    } else {
      for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
        const int c = CPOW2 ? (j & (C - 1)) : (j % C), r = CPOW2 ? (j >> lc) : (j / C);
        const int nl = r / T, t = r - nl * T;
        sm[fin_pad(nl * row + c * T + t)] += gp[j];
      }
    }
    si = s.next;
  }
}

__global__ void __launch_bounds__(256) finish_unpack_kernel(const FinSeg* __restrict__ segs, const int2* __restrict__ chunks,
                                                            const double* __restrict__ dots) {
  mtd_pdl_prologue();
  __shared__ float sm[kFinSmem];
  const int2 ck = chunks[blockIdx.x];
  const FinSeg head = segs[ck.x];
  const size_t total = (size_t)head.N * head.T * head.C;
  const size_t end = min(total, (size_t)ck.y + (size_t)fin_chunk_elems(head.T, head.C));
  if (fin_row_major(head)) {
    // Conv2d / Linear layout, whole packed rows: sums accumulated in shared memory at the element's REFERENCE position,
    // one coalesced store.  The (t, c) decomposition of the packed index is the inner loop of a 60-140 MB pass per
    // backward sweep, so it is compiled for the tap counts the model has (1, 9, 16: constant divisions) and uses shifts
    // for power-of-two channel counts.
    const int cnt = (int)(end - ck.y), T = (int)head.T, C = (int)head.C;
    const int n0 = (int)(ck.y / (size_t)(T * C));
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) sm[fin_pad(j)] = 0.f;
    __syncthreads();        // the accumulation below writes PERMUTED positions (another thread's j): zeroing must be complete
    const bool cpow2 = (C & (C - 1)) == 0;
    if (T == 9 && cpow2) fin_accumulate<9, true>(segs, ck, dots, sm, cnt, C, n0);
    else if (T == 16 && cpow2) fin_accumulate<16, true>(segs, ck, dots, sm, cnt, C, n0);
    else if (T == 1 && cpow2) fin_accumulate<1, true>(segs, ck, dots, sm, cnt, C, n0);
    else fin_accumulate<0, false>(segs, ck, dots, sm, cnt, C, n0);
    __syncthreads();
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) head.dw[ck.y + j] = sm[fin_pad(j)];
    return;
  }
  for (size_t i = (size_t)ck.y + threadIdx.x; i < end; i += blockDim.x) {
    const size_t ref = fin_ref_index(head, i);
    float sum = 0.f;
    long long si = ck.x;
    while (si >= 0) {
      const FinSeg& s = segs[si];
      float g = (s.flip & kFinNoGp) ? 0.f : s.gp[i];
      if (s.inv_sigma) {
        const float alpha = __ldg(s.inv_sigma);
        const float beta = s.dot_zw ? (float)(*s.dot_zw) : (float)dots[s.slot] * alpha;
        const size_t srow = ref / (size_t)s.sn_cols, col = ref - srow * (size_t)s.sn_cols;
        g = ((s.flip & kFinPrescaled) ? 1.f : alpha) * g - alpha * beta * __ldg(s.u + srow) * __ldg(s.v + col);
      }
      sum += g;
      si = s.next;
    }
    head.dw[ref] = sum;
  }
}

// Fill the (sN, sC, toff) mapping for a reference weight tensor.
//   transposed == 0: Conv2d / Linear layout (Cout, Cin, kh, kw)
//   transposed == 1: ConvTranspose2d layout (Cin, Cout, kh, kw), stride 1: the equivalent conv
//                    weight is W[co][ci][ky][kx] = Wt[ci][co][kh-1-ky][kw-1-kx]   (SURVEY A6)
// Forward orientation: n = co, c = ci, tap t = (ky, kx) with source offset (ky - pad, kx - pad).
void fwd_mapping(PackArgs& p, int transposed, int Cout, int Cin, int kh, int kw) {
  p.N = Cout; p.T = kh * kw; p.C = Cin;
  if (!transposed) {
    p.sN = (long long)Cin * kh * kw; p.sC = (long long)kh * kw;
    for (int t = 0; t < p.T; ++t) p.toff[t] = t;
  } else {
    p.sN = (long long)kh * kw; p.sC = (long long)Cout * kh * kw;
    for (int t = 0; t < p.T; ++t) p.toff[t] = p.T - 1 - t;
  }
}

// mtd_conv_pack_batch_begin / _end: between them every pack entry point RECORDS its work instead of launching it
// (host-side list, one batch at a time, not thread-safe); _end launches ceil(n / kPackBatch) batched kernels.
struct PackRec { const float* w; float* out; PackArgs p; };
static std::vector<PackRec>* g_pack_batch = nullptr;

int pack_launch(const float* w, float* out, const PackArgs& p, cudaStream_t st) {
  if (g_pack_batch) {
    g_pack_batch->push_back(PackRec{w, out, p});
    return MTD_OK;
  }
  size_t total = (size_t)p.N * p.T * p.C;
  int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)mtd_sm_count() * 16);
  mtd_launch(pack_weights_kernel, blocks, 256, 0, st, w, out, p);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// ---------------------------------------------------------------------------------------------
// weight gradient:  gp[n][t][c] = sum_p dz[p][n] * x[p@t][c]
// ---------------------------------------------------------------------------------------------
struct WgradArgs {
  const float* src1;
  const float* src2;
  int C1, C2;
  int B, H, W;
  const float* dz;
  int N, Ho, Wo;
  int T, sy, sx;
  int dy[kMaxTaps], dx[kMaxTaps];
  float* gp;
  int splits;
};

template <int TN, int TC, bool VEC>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const __grid_constant__ WgradArgs a) {
  mtd_pdl_prologue();
  constexpr int BN = 16 * TN, BC = 16 * TC, BK = 16;
  constexpr int A_Q = BN / 4, B_Q = BC / 4;                 // float4 slots per pixel row
  constexpr int A_PER = (BK * A_Q + 255) / 256, B_PER = (BK * B_Q + 255) / 256;
  __shared__ __align__(16) float As[2][BK][BN];
  __shared__ __align__(16) float Bs[2][BK][BC];

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n0 = blockIdx.x * BN, c0 = blockIdx.y * BC;
  const int t = blockIdx.z / a.splits, split = blockIdx.z - t * a.splits;
  const int Ctot = a.C1 + a.C2;
  const int HoWo = a.Ho * a.Wo;
  const int M = a.B * HoWo;
  const int per = (((M + a.splits - 1) / a.splits) + BK - 1) / BK * BK;
  const int p_begin = split * per, p_end = min(M, p_begin + per);
  if (p_begin >= p_end) return;
  const int nsteps = (p_end - p_begin + BK - 1) / BK;
  const int ddy = a.dy[t], ddx = a.dx[t];

  float4 ra[A_PER], rb[B_PER];
  auto load_tiles = [&](int step) {
    int pbase = p_begin + step * BK;
#pragma unroll
    for (int q = 0; q < A_PER; ++q) {
      int s = tid + q * 256;
      int prow = s / A_Q, nq = s - prow * A_Q;
      int p = pbase + prow;
      int n = n0 + nq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (prow < BK && p < p_end) {
        const float* row = a.dz + (size_t)p * a.N;
        if (VEC) { if (n < a.N) v = __ldg(reinterpret_cast<const float4*>(row + n)); }
        else {
          float tmp[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) tmp[j] = (n + j < a.N) ? __ldg(row + n + j) : 0.f;
          v = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
        }
      }
      ra[q] = v;
    }
#pragma unroll
    for (int q = 0; q < B_PER; ++q) {
      int s = tid + q * 256;
      int prow = s / B_Q, cq = s - prow * B_Q;
      int p = pbase + prow;
      int c = c0 + cq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (prow < BK && p < p_end) {
        int b = p / HoWo, r = p - b * HoWo;
        int oy = r / a.Wo, ox = r - oy * a.Wo;
        int iy = oy * a.sy + ddy, ix = ox * a.sx + ddx;
        if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W) {
          size_t pix = ((size_t)b * a.H + iy) * a.W + ix;
          if (VEC) {
            if (c < a.C1) v = __ldg(reinterpret_cast<const float4*>(a.src1 + pix * a.C1 + c));
            else if (c < Ctot) v = __ldg(reinterpret_cast<const float4*>(a.src2 + pix * a.C2 + (c - a.C1)));
          } else {
            float tmp[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              int cc = c + j;
              tmp[j] = cc < a.C1 ? __ldg(a.src1 + pix * a.C1 + cc)
                                 : (cc < Ctot ? __ldg(a.src2 + pix * a.C2 + (cc - a.C1)) : 0.f);
            }
            v = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
          }
        }
      }
      rb[q] = v;
    }
  };
  auto store_tiles = [&](int buf) {
#pragma unroll
    for (int q = 0; q < A_PER; ++q) {
      int s = tid + q * 256;
      int prow = s / A_Q, nq = s - prow * A_Q;
      if (prow < BK) *reinterpret_cast<float4*>(&As[buf][prow][nq * 4]) = ra[q];
    }
#pragma unroll
    for (int q = 0; q < B_PER; ++q) {
      int s = tid + q * 256;
      int prow = s / B_Q, cq = s - prow * B_Q;
      if (prow < BK) *reinterpret_cast<float4*>(&Bs[buf][prow][cq * 4]) = rb[q];
    }
  };

  float acc[TN][TC];
#pragma unroll
  for (int i = 0; i < TN; ++i)
#pragma unroll
    for (int j = 0; j < TC; ++j) acc[i][j] = 0.f;

  load_tiles(0);
  store_tiles(0);
  __syncthreads();
  int buf = 0;
  for (int step = 0; step < nsteps; ++step) {
    bool has_next = step + 1 < nsteps;
    if (has_next) load_tiles(step + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float av[TN], bv[TC];
#pragma unroll
      for (int i = 0; i < TN; ++i) av[i] = As[buf][k][ty * TN + i];
#pragma unroll
      for (int j = 0; j < TC; ++j) bv[j] = Bs[buf][k][tx * TC + j];
#pragma unroll
      for (int i = 0; i < TN; ++i)
#pragma unroll
        for (int j = 0; j < TC; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (has_next) store_tiles(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
#pragma unroll
  for (int i = 0; i < TN; ++i) {
    int n = n0 + ty * TN + i;
    if (n >= a.N) continue;
#pragma unroll
    for (int j = 0; j < TC; ++j) {
      int c = c0 + tx * TC + j;
      if (c >= Ctot) continue;
      float* dst = a.gp + ((size_t)n * a.T + t) * Ctot + c;
      if (a.splits > 1) atomicAdd(dst, acc[i][j]);
      else *dst = acc[i][j];
    }
  }
}

int launch_wgrad(WgradArgs& a, cudaStream_t st) {
  const int Ctot = a.C1 + a.C2;
  const int M = a.B * a.Ho * a.Wo;
  if (M <= 0 || a.N <= 0 || Ctot <= 0 || a.T <= 0 || a.T > kMaxTaps) return MTD_EINVAL;
  bool vec = (a.C1 % 4 == 0) && (a.C2 % 4 == 0) && (a.N % 4 == 0) && mtd_aligned16(a.src1) &&
             mtd_aligned16(a.dz) && (a.C2 == 0 || mtd_aligned16(a.src2));
  bool thin_n = a.N <= 16, thin_c = Ctot <= 16;
  int BN = thin_n ? 16 : 64, BC = thin_c ? 16 : 64;
  dim3 grid((a.N + BN - 1) / BN, (Ctot + BC - 1) / BC, a.T);
  int tiles = grid.x * grid.y * grid.z;
  int target = 4 * mtd_sm_count();
  int splits = 1;
  if (tiles < target) splits = std::min((target + tiles - 1) / tiles, std::max(1, M / 64));
  if (splits > 256) splits = 256;
  a.splits = splits;
  grid.z = a.T * splits;
  if (splits > 1) MTD_CUDA(cudaMemsetAsync(a.gp, 0, (size_t)a.N * a.T * Ctot * sizeof(float), st));
#define WG_LAUNCH(TN_, TC_)                                                              \
  do {                                                                                   \
    if (vec) mtd_launch(conv_wgrad_kernel<TN_, TC_, true>, grid, 256, 0, st, a);                 \
    else mtd_launch(conv_wgrad_kernel<TN_, TC_, false>, grid, 256, 0, st, a);                    \
  } while (0)
  if (thin_n && thin_c) WG_LAUNCH(1, 1);
  else if (thin_n) WG_LAUNCH(1, 4);
  else if (thin_c) WG_LAUNCH(4, 1);
  else WG_LAUNCH(4, 4);
#undef WG_LAUNCH
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// ---------------------------------------------------------------------------------------------
// dz = dy * act'(y)  (+ per-channel sums of dz accumulated into dbias, pre-zeroed by the caller
// wrapper).  (M, N) row-major, N = channels.
// ---------------------------------------------------------------------------------------------
// Fold outputs of mtd_act_bwd_acc (the FOLD instantiations below): dz of one backward pass is also folded into an
// accumulator that spans several passes, acc (+)= dz * scale[g], with zw[g] += sum dz . (y_pre - bias) per batched
// call g (see act_bwd_sn_kernel).  `group` counts elements (scalar kernel) or float4s (vector kernel) per call.
struct ActFold {
  float* acc;
  const float* scale;      // per-call 1/sigma, or null (scale 1)
  const float* bias;       // null: no bias
  double* zw;              // null: no <G, W~> accumulation
  size_t group;
  int first;               // 1: acc is written, 0: acc is read, added to and written
};

template <bool FOLD>
__global__ void act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dz,
                               float* __restrict__ dbias, size_t total, int N, int act, float slope, ActFold f) {
  mtd_pdl_prologue();
  extern __shared__ float colsum[];   // N floats when dbias != null
  if (dbias) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) colsum[i] = 0.f;
    __syncthreads();
  }
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  const bool fixed = dbias && (stride % (size_t)N == 0);   // channel of this thread never changes
  float priv = 0.f;
  double part[4] = {0.0, 0.0, 0.0, 0.0};                     // FOLD: up to 4 batched calls
  for (; i < total; i += stride) {
    float g = dy[i];
    if constexpr (FOLD) {
      const float t = (act != MTD_ACT_NONE || f.zw) ? __ldg(y + i) : 0.f;
      if (act != MTD_ACT_NONE) g *= mtd_act_grad(t, act, slope);
      const int gi = (i >= f.group) + (i >= 2 * f.group) + (i >= 3 * f.group);
      const float a = f.scale ? __ldg(f.scale + gi) : 1.f;
      f.acc[i] = f.first ? g * a : f.acc[i] + g * a;
      if (f.zw) {
        const float yp = (act == MTD_ACT_LEAKY && !(t > 0.f)) ? t * (1.f / slope) : t;
        part[gi] += (double)(g * (yp - (f.bias ? __ldg(f.bias + i % N) : 0.f)));
      }
    } else {
      if (act != MTD_ACT_NONE) g *= mtd_act_grad(__ldg(y + i), act, slope);
    }
    if (dz) dz[i] = g;
    if (dbias) {
      if (fixed) priv += g;
      else atomicAdd(&colsum[i % N], g);
    }
  }
  if (dbias) {
    if (fixed) {
      size_t first = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
      atomicAdd(&colsum[first % N], priv);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < N; c += blockDim.x) {
      float v = colsum[c];
      if (v != 0.f) atomicAdd(dbias + c, v);
    }
  }
  if constexpr (FOLD) {
    if (f.zw) {
      __shared__ double red[32];
      const int ngroups = (int)((total + f.group - 1) / f.group);
      for (int k = 0; k < ngroups && k < 4; ++k) {
        const double r = block_sum(part[k], red);
        if (threadIdx.x == 0 && r != 0.0) atomicAdd(f.zw + k, r);
      }
    }
  }
}

// float4 version (N % 4 == 0, 16-byte aligned pointers): 4 channels per thread; dy and y are read for the last
// time here (streaming loads), dz is re-read at once by dgrad / wgrad and stays in L2.
__global__ void __launch_bounds__(256) act_bwd_v4_kernel(const float4* __restrict__ dy, const float4* __restrict__ y,
                                                         float4* __restrict__ dz, float* __restrict__ dbias, size_t total4,
                                                         int N4, int act, float slope) {
  mtd_pdl_prologue();
  extern __shared__ float colsum[];   // 4 * N4 floats when dbias != null
  if (dbias) {
    for (int i = threadIdx.x; i < 4 * N4; i += blockDim.x) colsum[i] = 0.f;
    __syncthreads();
  }
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const bool fixed = dbias && (stride % (size_t)N4 == 0);   // channel group of this thread never changes
  float4 priv = make_float4(0.f, 0.f, 0.f, 0.f);
  const size_t first = i;
  for (; i < total4; i += stride) {
    float4 g = __ldcs(dy + i);
    if (act != MTD_ACT_NONE) {
      const float4 t = __ldcs(y + i);
      g.x *= mtd_act_grad(t.x, act, slope); g.y *= mtd_act_grad(t.y, act, slope);
      g.z *= mtd_act_grad(t.z, act, slope); g.w *= mtd_act_grad(t.w, act, slope);
    }
    if (dz) dz[i] = g;
    if (dbias) {
      if (fixed) { priv.x += g.x; priv.y += g.y; priv.z += g.z; priv.w += g.w; }
      else {
        float* cs = colsum + 4 * (i % N4);
        atomicAdd(cs, g.x); atomicAdd(cs + 1, g.y); atomicAdd(cs + 2, g.z); atomicAdd(cs + 3, g.w);
      }
    }
  }
  if (dbias) {
    if (fixed && first < total4) {
      float* cs = colsum + 4 * (first % N4);
      atomicAdd(cs, priv.x); atomicAdd(cs + 1, priv.y); atomicAdd(cs + 2, priv.z); atomicAdd(cs + 3, priv.w);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 4 * N4; c += blockDim.x) {
      float v = colsum[c];
      if (v != 0.f) atomicAdd(dbias + c, v);
    }
  }
}

// act_bwd for spectrally-normalised layers: additionally accumulates, per batched reference call g (a contiguous
// block of `group4` float4 elements), zw[g] = sum dz . (y_pre - bias): with y_pre = conv(x, W_orig)/sigma + bias this is
// <G_g, W_orig>/sigma_g = <G_g, W~_g>, the coefficient of the spectral-norm weight-gradient correction -- taken from data
// this pass reads anyway instead of a separate pass over the packed gradient and the weight.  LeakyReLU is inverted
// exactly (y_pre = y > 0 ? y : y / slope); not available for ReLU (y = 0 loses y_pre).  zw and dbias pre-zeroed.
// FOLD (mtd_act_bwd_acc): dz is written unscaled, dz * dz_scale[g] goes to acc (written when acc_first, else added),
// zw is optional and y may be null when act is none and zw is null.
template <bool FOLD>
__global__ void __launch_bounds__(256) act_bwd_sn_kernel(const float4* __restrict__ dy, const float4* __restrict__ y,
                                                         float4* __restrict__ dz, float* __restrict__ dbias,
                                                         const float4* __restrict__ bias, double* __restrict__ zw,
                                                         const float* __restrict__ dz_scale, size_t total4, size_t group4,
                                                         int N4, int act, float slope, float4* __restrict__ acc,
                                                         int acc_first) {
  mtd_pdl_prologue();
  extern __shared__ float colsum[];   // 4 * N4 floats when dbias != null
  __shared__ double red[32];
  if (dbias) {
    for (int i = threadIdx.x; i < 4 * N4; i += blockDim.x) colsum[i] = 0.f;
    __syncthreads();
  }
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;      // a multiple of N4 (host guarantees it): channels are fixed
  const size_t first = i;
  const float4 b4 = (bias && first < total4) ? __ldg(bias + first % N4) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float inv_slope = 1.f / slope;
  float4 priv = make_float4(0.f, 0.f, 0.f, 0.f);
  double part[4] = {0.0, 0.0, 0.0, 0.0};                     // up to 4 batched calls
  for (; i < total4; i += stride) {
    float4 g = __ldcs(dy + i);
    const float4 t = (FOLD && !y) ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldcs(y + i);
    float4 yp = t;
    if (act == MTD_ACT_LEAKY) {
      g.x *= t.x > 0.f ? 1.f : slope; g.y *= t.y > 0.f ? 1.f : slope; g.z *= t.z > 0.f ? 1.f : slope; g.w *= t.w > 0.f ? 1.f : slope;
      yp.x = t.x > 0.f ? t.x : t.x * inv_slope; yp.y = t.y > 0.f ? t.y : t.y * inv_slope;
      yp.z = t.z > 0.f ? t.z : t.z * inv_slope; yp.w = t.w > 0.f ? t.w : t.w * inv_slope;
    }
    const int gi = (i >= group4) + (i >= 2 * group4) + (i >= 3 * group4);      // groups <= 4
    if constexpr (FOLD) {
      if (dz) dz[i] = g;
      const float a = dz_scale ? __ldg(dz_scale + gi) : 1.f;
      const float4 s = make_float4(g.x * a, g.y * a, g.z * a, g.w * a);
      if (acc_first) {
        acc[i] = s;
      } else {
        const float4 o = acc[i];
        acc[i] = make_float4(o.x + s.x, o.y + s.y, o.z + s.z, o.w + s.w);
      }
    } else if (dz) {
      // dz_scale: write dz / sigma_g, so that dgrad needs no epilogue scale and ONE weight-gradient GEMM over the
      // whole batch yields sum_g G_g / sigma_g; the bias gradient and zw use the unscaled dz
      const float a = dz_scale ? __ldg(dz_scale + gi) : 1.f;
      dz[i] = make_float4(g.x * a, g.y * a, g.z * a, g.w * a);
    }
    priv.x += g.x; priv.y += g.y; priv.z += g.z; priv.w += g.w;
    if (!FOLD || zw) {
      const float d = g.x * (yp.x - b4.x) + g.y * (yp.y - b4.y) + g.z * (yp.z - b4.z) + g.w * (yp.w - b4.w);
      part[gi] += (double)d;
    }
  }
  if (dbias) {
    if (first < total4) {
      float* cs = colsum + 4 * (first % N4);
      atomicAdd(cs, priv.x); atomicAdd(cs + 1, priv.y); atomicAdd(cs + 2, priv.z); atomicAdd(cs + 3, priv.w);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 4 * N4; c += blockDim.x) {
      float v = colsum[c];
      if (v != 0.f) atomicAdd(dbias + c, v);
    }
  }
  if (FOLD && !zw) return;
  const int ngroups = (int)((total4 + group4 - 1) / group4);
  for (int k = 0; k < ngroups && k < 4; ++k) {
    const double r = block_sum(part[k], red);
    if (threadIdx.x == 0 && r != 0.0) atomicAdd(zw + k, r);
  }
}

void tap_table_fwd(int* dy, int* dx, int kh, int kw, int pad) {
  for (int ky = 0; ky < kh; ++ky)
    for (int kx = 0; kx < kw; ++kx) {
      dy[ky * kw + kx] = ky - pad;
      dx[ky * kw + kx] = kx - pad;
    }
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

static int g_pack_blocked = 0;     // set by the *_blocked entry points around the shared implementation
static int g_pack_tf32 = 0;

int mtd_conv_pack_fwd(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, float* out, void* stream) {
  MTD_REQUIRE(w_ref && out && Cout > 0 && Cin > 0 && kh > 0 && kw > 0 && kh * kw <= kMaxTaps);
  PackArgs p;
  fwd_mapping(p, transposed, Cout, Cin, kh, kw);
  p.blocked = g_pack_blocked; p.tf32 = g_pack_tf32; p.lo_off = (long long)Cout * Cin * kh * kw;
  if (p.blocked) MTD_REQUIRE(Cout % 32 == 0 && Cin % 32 == 0);
  return pack_launch(w_ref, out, p, (cudaStream_t)stream);
}

// dgrad packing.  stride 1: out[ci][t][co] with t = ky*kw+kx (source offset pad-ky, pad-kx).
// stride 2 (4x4, pad 1 only): out[cls][ci][t2][co], cls = py*2+px, t2 = a*2+b where
// ky = (1-py) + 2a, kx = (1-px) + 2b.
int mtd_conv_pack_dgrad(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int stride, float* out,
                        void* stream) {
  MTD_REQUIRE(w_ref && out && Cout > 0 && Cin > 0 && kh * kw <= kMaxTaps);
  PackArgs f;
  fwd_mapping(f, transposed, Cout, Cin, kh, kw);
  cudaStream_t st = (cudaStream_t)stream;
  if (stride == 1) {
    PackArgs p;
    p.N = Cin; p.T = kh * kw; p.C = Cout; p.sN = f.sC; p.sC = f.sN;
    for (int t = 0; t < p.T; ++t) p.toff[t] = f.toff[t];
    p.blocked = g_pack_blocked; p.tf32 = g_pack_tf32; p.lo_off = (long long)Cout * Cin * kh * kw;
    if (p.blocked) MTD_REQUIRE(Cout % 32 == 0 && Cin % 32 == 0);
    return pack_launch(w_ref, out, p, st);
  }
  MTD_REQUIRE(stride == 2 && kh == 4 && kw == 4 && !transposed);
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      PackArgs p;
      p.blocked = g_pack_blocked; p.tf32 = g_pack_tf32; p.lo_off = (long long)Cout * Cin * kh * kw;
      if (p.blocked) MTD_REQUIRE(Cout % 32 == 0 && Cin % 32 == 0);
      p.N = Cin; p.T = 4; p.C = Cout; p.sN = f.sC; p.sC = f.sN;
      for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b) {
          int ky = (1 - py) + 2 * a, kx = (1 - px) + 2 * b;
          p.toff[a * 2 + b] = f.toff[ky * kw + kx];
        }
      int rc = pack_launch(w_ref, out + (size_t)(py * 2 + px) * Cin * 4 * Cout, p, st);
      if (rc) return rc;
    }
  return MTD_OK;
}

// Same packs in the tile-major layout the tensor-core kernels read: [rows/32][K/32][32][32] (rows = Cout for the
// forward pack, Cin for dgrad; K = taps x channels), with the TF32 operand preparation fused in: tf32 = 0 plain
// copy, 1 rounded to nearest tf32, 3 [hi | lo] halves for the 3xTF32 mode (`out` then holds 2 x numel floats).
// Requires Cout % 32 == 0 and Cin % 32 == 0.
int mtd_conv_pack_fwd_blocked(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int tf32, float* out,
                              void* stream) {
  MTD_REQUIRE(tf32 == 0 || tf32 == 1 || tf32 == 3);
  g_pack_blocked = 1; g_pack_tf32 = tf32;
  int rc = mtd_conv_pack_fwd(w_ref, transposed, Cout, Cin, kh, kw, out, stream);
  g_pack_blocked = 0; g_pack_tf32 = 0;
  return rc;
}
int mtd_conv_pack_dgrad_blocked(const float* w_ref, int transposed, int Cout, int Cin, int kh, int kw, int stride, int tf32,
                                float* out, void* stream) {
  MTD_REQUIRE(tf32 == 0 || tf32 == 1 || tf32 == 3);
  g_pack_blocked = 1; g_pack_tf32 = tf32;
  int rc = mtd_conv_pack_dgrad(w_ref, transposed, Cout, Cin, kh, kw, stride, out, stream);
  g_pack_blocked = 0; g_pack_tf32 = 0;
  return rc;
}

int mtd_conv_pack_batch_begin(void) {
  MTD_REQUIRE(g_pack_batch == nullptr);
  g_pack_batch = new std::vector<PackRec>();
  return MTD_OK;
}

// Launches everything recorded since mtd_conv_pack_batch_begin: kPackBatch packs per kernel.
int mtd_conv_pack_batch_end(void* stream) {
  MTD_REQUIRE(g_pack_batch != nullptr);
  std::vector<PackRec>* recs = g_pack_batch;
  g_pack_batch = nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = MTD_OK;
  for (size_t i0 = 0; i0 < recs->size() && rc == MTD_OK; i0 += kPackBatch) {
    PackBatch pb;
    memset(&pb, 0, sizeof(pb));
    pb.n = (int)std::min<size_t>(kPackBatch, recs->size() - i0);
    int blocks = 0;
    for (int k = 0; k < pb.n; ++k) {
      const PackRec& r = (*recs)[i0 + k];
      pb.w[k] = r.w; pb.out[k] = r.out; pb.p[k] = r.p;
      pb.first_block[k] = blocks;
      const size_t total = (size_t)r.p.N * r.p.T * r.p.C;
      blocks += (int)((total + kPackChunk - 1) / kPackChunk);
    }
    pb.first_block[pb.n] = blocks;
    mtd_launch(pack_batched_kernel, blocks, 256, 0, st, pb);
    ++g_mtd_kernel_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = (int)e;
  }
  delete recs;
  return rc;
}

int mtd_conv_fwd(const float* x1, const float* x2, const float* wp, const float* bias, const float* scale, int scale_group,
                 float* y,
                 float* aux, const float* add1, const float* add2, int B, int H, int W, int C1, int C2, int N, int kh,
                 int kw, int stride, int pad, int pre_act, int post_act, float slope, void* stream) {
  MTD_REQUIRE(x1 && wp && y && B > 0 && H > 0 && W > 0 && C1 > 0 && C2 >= 0 && N > 0);
  MTD_REQUIRE((C2 == 0) == (x2 == nullptr));
  MTD_REQUIRE(stride >= 1 && kh * kw <= kMaxTaps);
  ConvArgs a{};
  a.src1 = x1; a.src2 = x2; a.C1 = C1; a.C2 = C2; a.B = B; a.H = H; a.W = W;
  a.wp = wp; a.N = N; a.T = kh * kw;
  a.Ho = (H + 2 * pad - kh) / stride + 1;
  a.Wo = (W + 2 * pad - kw) / stride + 1;
  MTD_REQUIRE(a.Ho > 0 && a.Wo > 0);
  a.sy = a.sx = stride;
  tap_table_fwd(a.dy, a.dx, kh, kw, pad);
  a.out = y; a.outH = a.Ho; a.outW = a.Wo; a.omy = a.omx = 1; a.ooy = a.oox = 0;
  a.scale = scale; a.bias = bias; a.pre_act = pre_act; a.add1 = add1; a.add2 = add2; a.post_act = post_act;
  a.scale_span = (scale && scale_group > 0 && scale_group < B) ? (long long)scale_group * a.Ho * a.Wo * N : 0;
  a.mask_src = nullptr; a.mask_act = 0; a.slope = slope; a.aux = aux;
  return launch_conv(a, (cudaStream_t)stream);
}

// dx (B,H,W,Cin) = scale * dgrad(dz (B,Ho,Wo,Cout)) [+ add1 + add2] [* act'(mask_src)]
int mtd_conv_dgrad(const float* dz, const float* wpd, float* dx, const float* scale, int scale_group, const float* add1,
                   const float* add2, const float* mask_src, int mask_act, float slope, int B, int H, int W, int Cin,
                   int Cout, int kh, int kw, int stride, int pad, void* stream) {
  MTD_REQUIRE(dz && wpd && dx && B > 0 && Cin > 0 && Cout > 0 && kh * kw <= kMaxTaps);
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  ConvArgs a{};
  a.src1 = dz; a.src2 = nullptr; a.C1 = Cout; a.C2 = 0; a.B = B; a.H = Ho; a.W = Wo;
  a.N = Cin;
  a.out = dx; a.outH = H; a.outW = W;
  a.scale = scale; a.bias = nullptr; a.pre_act = 0; a.add1 = add1; a.add2 = add2; a.post_act = 0;
  a.scale_span = (scale && scale_group > 0 && scale_group < B) ? (long long)scale_group * H * W * Cin : 0;
  a.mask_src = mask_src; a.mask_act = mask_act; a.slope = slope; a.aux = nullptr;
  if (stride == 1) {
    a.wp = wpd; a.T = kh * kw; a.Ho = H; a.Wo = W; a.sy = a.sx = 1;
    for (int ky = 0; ky < kh; ++ky)
      for (int kx = 0; kx < kw; ++kx) {
        a.dy[ky * kw + kx] = pad - ky;
        a.dx[ky * kw + kx] = pad - kx;
      }
    a.omy = a.omx = 1; a.ooy = a.oox = 0;
    return launch_conv(a, (cudaStream_t)stream);
  }
  MTD_REQUIRE(stride == 2 && kh == 4 && kw == 4 && pad == 1 && H % 2 == 0 && W % 2 == 0);
  // y = 2i+py receives ky with (py+1-ky) even: ky = (1-py)+2a, source row i + (py+1-ky)/2
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      ConvArgs c = a;
      c.wp = wpd + (size_t)(py * 2 + px) * Cin * 4 * Cout;
      c.T = 4; c.Ho = H / 2; c.Wo = W / 2; c.sy = c.sx = 1;
      for (int aa = 0; aa < 2; ++aa)
        for (int bb = 0; bb < 2; ++bb) {
          int ky = (1 - py) + 2 * aa, kx = (1 - px) + 2 * bb;
          c.dy[aa * 2 + bb] = (py + 1 - ky) / 2;
          c.dx[aa * 2 + bb] = (px + 1 - kx) / 2;
        }
      c.omy = c.omx = 2; c.ooy = py; c.oox = px;
      int rc = launch_conv(c, (cudaStream_t)stream);
      if (rc) return rc;
    }
  return MTD_OK;
}

// gp[N][T][C1+C2] = sum over pixels dz x (packed, forward orientation).
int mtd_conv_wgrad(const float* x1, const float* x2, const float* dz, float* gp, int B, int H, int W, int C1, int C2,
                   int N, int kh, int kw, int stride, int pad, void* stream) {
  MTD_REQUIRE(x1 && dz && gp && B > 0 && C1 > 0 && C2 >= 0 && N > 0 && kh * kw <= kMaxTaps);
  MTD_REQUIRE((C2 == 0) == (x2 == nullptr));
  WgradArgs a{};
  a.src1 = x1; a.src2 = x2; a.C1 = C1; a.C2 = C2; a.B = B; a.H = H; a.W = W;
  a.dz = dz; a.N = N;
  a.Ho = (H + 2 * pad - kh) / stride + 1;
  a.Wo = (W + 2 * pad - kw) / stride + 1;
  a.T = kh * kw; a.sy = a.sx = stride;
  tap_table_fwd(a.dy, a.dx, kh, kw, pad);
  a.gp = gp;
  const int Ctot = C1 + C2;
  if (stride == 1 && a.Ho == H && a.Wo == W && (N == 1 || Ctot == 1) && (N == 1 ? Ctot : N) <= 256) {
    // thin layer: gp[n][t][c] with n == 0 (vector = x, scalar = dz, x pixel = p + tap  =>  s index = q - tap for q over x)
    // or c == 0 (vector = dz, scalar = x at p + tap)
    cudaStream_t st = (cudaStream_t)stream;
    ThinWgArgs w{};
    w.B = B; w.H = H; w.W = W; w.T = a.T; w.out = gp;
    if (N == 1 && Ctot > 1) {
      w.V1 = x1; w.V2 = x2; w.J1 = C1; w.J2 = C2; w.s = dz;
      for (int t = 0; t < a.T; ++t) { w.dy[t] = -a.dy[t]; w.dx[t] = -a.dx[t]; }
      w.st_t = Ctot; w.st_j = 1;
    } else {
      w.V1 = dz; w.V2 = nullptr; w.J1 = N; w.J2 = 0; w.s = x1;
      for (int t = 0; t < a.T; ++t) { w.dy[t] = a.dy[t]; w.dx[t] = a.dx[t]; }
      w.st_t = Ctot; w.st_j = (long long)a.T * Ctot;          // Ctot == 1
    }
    const long long M = (long long)B * H * W;
    int blocks = mtd_sm_count() * 4;
    if (blocks > M / 64 + 1) blocks = (int)(M / 64 + 1);
    w.pix_per_block = (int)((M + blocks - 1) / blocks);
    blocks = (int)((M + w.pix_per_block - 1) / w.pix_per_block);
    MTD_CUDA(cudaMemsetAsync(gp, 0, (size_t)N * a.T * Ctot * sizeof(float), st));
    const int J = w.J1 + w.J2;
    const bool vec4 = (w.J1 % 4 == 0) && (w.J2 % 4 == 0) && J >= 4 && mtd_aligned16(w.V1) && (!w.V2 || mtd_aligned16(w.V2));
    const size_t smem = (size_t)a.T * J * sizeof(float);
    if (vec4) mtd_launch(thin_wgrad_kernel<true>, blocks, 256, smem, st, w);
    else mtd_launch(thin_wgrad_kernel<false>, blocks, 256, smem, st, w);
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
  return launch_wgrad(a, (cudaStream_t)stream);
}

// dw_ref (reference layout) from packed gp; spectral-norm correction when inv_sigma != null:
//   dW_orig = (G - <G, W~> u v^T) / sigma,  W~ = W_orig / sigma        (SURVEY A5)
// `scratch` = 8 bytes (double) + 4 bytes (float) of device workspace.
int mtd_conv_wgrad_finish(const float* gp, float* dw_ref, int transposed, int Cout, int Cin, int kh, int kw,
                          const float* w_ref, const float* u, const float* v, const float* inv_sigma, void* scratch,
                          void* stream) {
  MTD_REQUIRE(gp && dw_ref && Cout > 0 && Cin > 0 && kh * kw <= kMaxTaps);
  cudaStream_t st = (cudaStream_t)stream;
  UnpackArgs a{};
  fwd_mapping(a.p, transposed, Cout, Cin, kh, kw);
  size_t total = (size_t)Cout * Cin * kh * kw;
  int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)mtd_sm_count() * 16);
  if (inv_sigma) {
    MTD_REQUIRE(w_ref && u && v && scratch && !transposed);
    double* acc = (double*)scratch;
    MTD_CUDA(cudaMemsetAsync(acc, 0, 8, st));
    mtd_launch(dot_packed_ref_kernel, blocks, 256, 0, st, gp, w_ref, acc, a.p);
    MTD_CHECK_LAUNCH();
    a.inv_sigma = inv_sigma; a.dotgw = acc; a.u = u; a.v = v;
    a.sn_rows = Cout; a.sn_cols = (long long)Cin * kh * kw;
  }
  mtd_launch(unpack_grad_kernel, blocks, 256, 0, st, gp, dw_ref, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// Grid of the scalar act_bwd kernel: with column sums, the grid stride is made a multiple of N when possible (N is a
// power of two for every layer here), so that each thread's channel never changes.
static int act_bwd_scalar_blocks(size_t total, int N, bool colsums) {
  int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)mtd_sm_count() * 8);
  if (colsums) {
    size_t stride = (size_t)blocks * 256;
    if (stride % N != 0 && (size_t)N <= stride) {
      size_t s2 = stride / N * N;
      if (s2 % 256 == 0 && s2 > 0) blocks = (int)(s2 / 256);
    } else if ((size_t)N > stride) {
      blocks = (N + 255) / 256;
    }
  }
  return blocks;
}

// Grid of act_bwd_sn_kernel: its grid stride must be a multiple of N4 (fixed channels per thread); 0 if impossible.
static int act_bwd_sn_blocks(size_t total4, int N4) {
  int blocks = (int)std::min<size_t>((total4 + 255) / 256, (size_t)mtd_sm_count() * 4);
  size_t stride = (size_t)blocks * 256;
  if ((size_t)N4 > stride) blocks = (N4 + 255) / 256;
  else if (stride % N4 != 0) {
    size_t s2 = stride / N4 * N4;
    while (s2 > 0 && s2 % 256 != 0) s2 -= N4;
    blocks = (int)(s2 / 256);
  }
  return ((size_t)blocks * 256) % N4 == 0 ? blocks : 0;
}

// dz = dy * act'(y); dbias[N] (optional) = column sums of dz.  dz may be null (colsum only) and may
// alias dy.  dbias_zeroed != 0: the caller guarantees dbias is already all zero (e.g. carved from one zeroed slab
// per backward pass), which saves a memset node per layer.
int mtd_act_bwd(const float* dy, const float* y, float* dz, float* dbias, int dbias_zeroed, long long M, int N, int act,
                float slope, void* stream) {
  MTD_REQUIRE(dy && M > 0 && N > 0 && (act == MTD_ACT_NONE || y));
  cudaStream_t st = (cudaStream_t)stream;
  size_t total = (size_t)M * N;
  if (N % 4 == 0 && mtd_aligned16(dy) && (!y || mtd_aligned16(y)) && (!dz || mtd_aligned16(dz))) {
    const size_t total4 = total / 4;
    const int N4 = N / 4;
    int blocks = (int)std::min<size_t>((total4 + 255) / 256, (size_t)mtd_sm_count() * 4);
    if (dbias) {
      MTD_REQUIRE(N <= 8192);
      if (!dbias_zeroed) MTD_CUDA(cudaMemsetAsync(dbias, 0, (size_t)N * sizeof(float), st));
      // grid stride a multiple of the channel groups when possible (N is a power of two for every layer here)
      size_t stride = (size_t)blocks * 256;
      if (stride % N4 != 0 && (size_t)N4 <= stride) {
        size_t s2 = stride / N4 * N4;
        if (s2 % 256 == 0 && s2 > 0) blocks = (int)(s2 / 256);
      } else if ((size_t)N4 > stride) {
        blocks = (N4 + 255) / 256;
      }
    }
    mtd_launch(act_bwd_v4_kernel, blocks, 256, dbias ? N * sizeof(float) : 0, st, reinterpret_cast<const float4*>(dy),
               reinterpret_cast<const float4*>(y), reinterpret_cast<float4*>(dz), dbias, total4, N4, act, slope);
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
  if (dbias) {
    MTD_REQUIRE(N <= 8192);
    if (!dbias_zeroed) MTD_CUDA(cudaMemsetAsync(dbias, 0, (size_t)N * sizeof(float), st));
  }
  mtd_launch(act_bwd_kernel<false>, act_bwd_scalar_blocks(total, N, dbias != nullptr), 256, dbias ? N * sizeof(float) : 0, st,
             dy, y, dz, dbias, total, N, act, slope, ActFold{});
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// mtd_act_bwd for a spectrally-normalised layer whose batch holds `groups` (<= 4) reference calls of M/groups rows:
// also accumulates zw[g] += sum over group g of dz . (y_pre - bias) (see act_bwd_sn_kernel).  dbias (optional) and zw
// must be all zero on entry.  dz_scale (optional, `groups` floats = 1/sigma_g): the dz written is dz / sigma_g.  act: MTD_ACT_NONE or MTD_ACT_LEAKY.  Requires N % 4 == 0 and a power-of-two N <= 8192.
int mtd_act_bwd_sn(const float* dy, const float* y, float* dz, float* dbias, const float* bias, double* zw,
                   const float* dz_scale, int groups, long long M, int N, int act, float slope, void* stream) {
  MTD_REQUIRE(dy && y && zw && M > 0 && N > 0 && N % 4 == 0 && N <= 8192 && groups >= 1 && groups <= 4 && M % groups == 0);
  MTD_REQUIRE(act == MTD_ACT_NONE || act == MTD_ACT_LEAKY);
  MTD_REQUIRE(mtd_aligned16(dy) && mtd_aligned16(y) && (!dz || mtd_aligned16(dz)) && (!bias || mtd_aligned16(bias)));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t total4 = (size_t)M * N / 4;
  const int N4 = N / 4;
  const int blocks = act_bwd_sn_blocks(total4, N4);
  MTD_REQUIRE(blocks > 0);
  mtd_launch(act_bwd_sn_kernel<false>, blocks, 256, dbias ? N * sizeof(float) : 0, st, reinterpret_cast<const float4*>(dy),
             reinterpret_cast<const float4*>(y), reinterpret_cast<float4*>(dz), dbias, reinterpret_cast<const float4*>(bias), zw,
             dz_scale, total4, total4 / groups, N4, act, slope, static_cast<float4*>(nullptr), 0);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// One backward pass's activation backward that also folds dz into accumulators spanning several passes (see the
// header).  Same dz as mtd_act_bwd; N % 4 == 0 with 16-byte aligned operands takes the float4 kernel, anything else
// the scalar one.
int mtd_act_bwd_acc(const float* dy, const float* y, float* dz, float* acc, int acc_first, float* dbias, const float* bias,
                    double* zw, const float* inv_sigma, int groups, long long M, int N, int act, float slope, void* stream) {
  MTD_REQUIRE(dy && acc && M > 0 && N > 0 && N <= 8192 && groups >= 1 && groups <= 4 && M % groups == 0);
  MTD_REQUIRE(y || (act == MTD_ACT_NONE && !zw));
  MTD_REQUIRE(!zw || act == MTD_ACT_NONE || act == MTD_ACT_LEAKY);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t total = (size_t)M * N;
  if (N % 4 == 0 && mtd_aligned16(dy) && mtd_aligned16(acc) && (!y || mtd_aligned16(y)) && (!dz || mtd_aligned16(dz)) &&
      (!bias || mtd_aligned16(bias))) {
    const size_t total4 = total / 4;
    const int N4 = N / 4;
    const int blocks = act_bwd_sn_blocks(total4, N4);
    MTD_REQUIRE(blocks > 0);
    mtd_launch(act_bwd_sn_kernel<true>, blocks, 256, dbias ? N * sizeof(float) : 0, st, reinterpret_cast<const float4*>(dy),
               reinterpret_cast<const float4*>(y), reinterpret_cast<float4*>(dz), dbias, reinterpret_cast<const float4*>(bias),
               zw, inv_sigma, total4, total4 / groups, N4, act, slope, reinterpret_cast<float4*>(acc), acc_first);
  } else {
    const ActFold f{acc, inv_sigma, bias, zw, total / groups, acc_first};
    mtd_launch(act_bwd_kernel<true>, act_bwd_scalar_blocks(total, N, dbias != nullptr), 256, dbias ? N * sizeof(float) : 0,
               st, dy, y, dz, dbias, total, N, act, slope, f);
  }
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int mtd_wgrad_finish_chunk_elems(int taps, int cin) { return (int)fin_chunk_elems(taps, cin); }

// Batched form of mtd_conv_wgrad_finish (same arithmetic).  dots: n_segs doubles of device scratch (zeroed here).
int mtd_wgrad_finish_batched(const void* seg_tab, int n_segs, const void* dot_chunks, int n_dot_chunks, const void* head_chunks,
                             int n_head_chunks, double* dots, void* stream) {
  MTD_REQUIRE(seg_tab && head_chunks && dots && n_segs > 0 && n_head_chunks > 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_dot_chunks > 0) {
    MTD_REQUIRE(dot_chunks);
    MTD_CUDA(cudaMemsetAsync(dots, 0, (size_t)n_segs * sizeof(double), st));
    mtd_launch(finish_dot_kernel, n_dot_chunks, 256, 0, st, reinterpret_cast<const FinSeg*>(seg_tab),
                                                    reinterpret_cast<const int2*>(dot_chunks), dots);
    MTD_CHECK_LAUNCH();
  }
  mtd_launch(finish_unpack_kernel, n_head_chunks, 256, 0, st, reinterpret_cast<const FinSeg*>(seg_tab),
                                                      reinterpret_cast<const int2*>(head_chunks), dots);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

}  // extern "C"
