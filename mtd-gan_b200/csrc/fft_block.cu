// Frequency branch of the Res-FFT-Conv block, NHWC fp32 (C = 32 channels).
//
//   rfft2(ortho) -> cat[Re,Im] -> 1x1 conv (2C x 2C) + bias + ReLU -> complex -> irfft2(ortho)
//   (arch/Ours/networks.py:24-29), decomposed as
//     P1  fft_rows_fwd     : real FFT along W of every (b,h) row, two channels packed per complex
//                            transform; writes the half spectrum  X1[b][kw][h][c]  (complex)
//     P2  fft_cols_mix     : one CTA per (b,kw): complex FFT along H, per-frequency channel mix + bias + ReLU,
//                            inverse FFT along H -> X3[b][kw][h][c]
//     P3  fft_rows_inv     : half-spectrum inverse along W (Im of columns kw=0 and kw=W/2 dropped,
//                            SURVEY A1) fused with the block's residual adds  out = fft + add1 + add2
//   Backward (SURVEY A2/A3): P1 on the incoming gradient, fft_cols_mix_bwd (recomputes the ReLU mask
//   from the saved X1, accumulates dW/db partials with the column weights w_k, applies M^T), then P3.
//
// Every transform is a four-step FFT (fft_core.cuh): two register-resident radix-2 networks of N1 and N2 points
// around ONE shared-memory exchange, instead of log2(N) barrier-separated shared-memory passes:
//   * rows: the (q, n2) thread loads its N1 points straight from global memory (16 channel pairs x 2 positions =
//     256 contiguous bytes per warp load), so the input never passes through shared memory; the exchange buffer is
//     written in place and read strided; the real-pair separation  A_k = (Z_k + conj Z_{N-k})/2  takes Z_{N-k} from
//     the partner lane with ONE warp shuffle (threads k1 and N1-k1 of a channel pair are lanes l and l^16);
//   * columns: lane = channel, so every shared-memory access is a 256-byte row (conflict-free); the spectrum stays
//     in [k1][k2] order between the forward and the inverse transform -- the channel mix is frequency-local, so no
//     reordering pass exists.
// Lengths 64, 128, 256, 512 run these kernels (8x8, 8x16, 16x16, 16x32).  Every other length 1 <= N <= 512 runs the
// Bluestein kernels further down (forward only): P1 / P3 as one chirp-z transform per image row, P2 split into a
// column transform, a flat channel-mix pass and an inverse column transform.
#include <algorithm>
#include <cmath>
#include <mutex>
#include <vector>
#include "common.cuh"
#include "fft_core.cuh"
#include "mtdgan_b200.h"

namespace {

using namespace mtdfft;

constexpr int kC = 32, kC2 = 64, kQ = 16;          // channels, mix width, channel pairs (complex sequences per row)
constexpr int kThreadsFft = 256;

// tw[k] = exp(-2*pi*i*k/N), k < N (full circle: indexed with (n2*k1) mod N)
__device__ __forceinline__ void fill_twiddles(float2* tw, int N) {
  for (int k = threadIdx.x; k < N; k += blockDim.x) {
    float s, c;
    sincospif(-2.0f * (float)k / (float)N, &s, &c);
    tw[k] = make_float2(c, s);
  }
}

__device__ __forceinline__ float2 shfl_xor2(float2 v, int m) {
  return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}

// rows handled per CTA pass: two when both steps of a row need <= 128 threads (W = 64)
template <int N1, int N2>
struct RowsCfg {
  static constexpr int N = N1 * N2;
  static constexpr int IA = kQ * N2;                 // step-A items per row: (n2, q)
  static constexpr int IB = kQ * N1;                 // step-B items per row: (k1, q), warp = the pair {k1, N1-k1}
  static constexpr int RPB = (IA <= 128 && IB <= 128) ? 2 : 1;
  static constexpr size_t smem = (size_t)RPB * N * kQ * 8 + (size_t)N * 8;
};

// k1 of step-B lane: warp w of a row holds k1 = w (lanes 0-15) and N1 - w (lanes 16-31); warp 0 holds the two
// self-conjugate residues 0 and N1/2
template <int N1>
__device__ __forceinline__ int pair_k1(int w, int s) { return w == 0 ? (s ? N1 / 2 : 0) : (s ? N1 - w : w); }

// ------------------------------------------------------------------------------------------------
// P1: rows forward.  grid = ceil(B*H / RPB)
// ------------------------------------------------------------------------------------------------
template <int N1, int N2>
__global__ void __launch_bounds__(kThreadsFft) fft_rows_fwd_kernel(const float* __restrict__ x, float2* __restrict__ spec,
                                                                 int H, int nrows) {
  mtd_pdl_prologue();
  using Cfg = RowsCfg<N1, N2>;
  constexpr int N = Cfg::N, Wh = N / 2 + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* T = reinterpret_cast<float2*>(smem_raw);                 // [RPB][k1][n2][q]
  float2* tw = T + (size_t)Cfg::RPB * N * kQ;
  fill_twiddles(tw, N);
  __syncthreads();
  // ---- step A: N1-point FFTs over n1 of x[N2*n1 + n2], straight from global memory
  for (int it = threadIdx.x; it < Cfg::RPB * Cfg::IA; it += kThreadsFft) {
    const int r = it / Cfg::IA, rem = it - r * Cfg::IA;
    const int n2 = rem >> 4, q = rem & 15;
    const long long row = (long long)blockIdx.x * Cfg::RPB + r;
    if (row >= nrows) continue;
    const float2* src = reinterpret_cast<const float2*>(x + (size_t)row * N * kC) + q;
    float2 v[N1];
#pragma unroll
    for (int n1 = 0; n1 < N1; ++n1) v[n1] = __ldg(src + (size_t)(N2 * n1 + n2) * kQ);
    fft_reg<N1, false>(v);
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int k1 = brev_c(i, N1);
      const float2 w = tw[(n2 * k1) & (N - 1)];
      T[((r * N1 + k1) * N2 + n2) * kQ + q] = k1 == 0 ? v[i] : cmul(v[i], w);
    }
  }
  __syncthreads();
  // ---- step B: N2-point FFTs over n2; real-pair separation with the partner lane; store the half spectrum
  const float sc = rsqrtf((float)N) * 0.5f;
  for (int it = threadIdx.x; it < Cfg::RPB * Cfg::IB; it += kThreadsFft) {
    const int r = it / Cfg::IB, rem = it - r * Cfg::IB;
    const int w = rem >> 5, lane = rem & 31, s = lane >> 4, q = lane & 15;
    const long long row = (long long)blockIdx.x * Cfg::RPB + r;
    if (row >= nrows) continue;                       // warp-uniform (IB is a multiple of 32)
    const int k1 = pair_k1<N1>(w, s);
    float2 v[N2];
#pragma unroll
    for (int n2 = 0; n2 < N2; ++n2) v[n2] = T[((r * N1 + k1) * N2 + n2) * kQ + q];
    fft_reg<N2, false>(v);                            // v[j] = Z[k1 + N1 * brev(j)]
    const int b = (int)(row / H), h = (int)(row - (long long)b * H);
    float2* dst0 = spec + ((size_t)b * Wh * H + h) * kC + 2 * q;
#pragma unroll
    for (int j = 0; j < N2; ++j) {
      const int k2 = brev_c(j, N2);
      if (k2 > N2 / 2) continue;
      if (k2 == N2 / 2 && w != 0) continue;           // k = N/2 exists only for k1 = 0
      const float2 own1 = v[N2 - 1 - j];              // Z[k1 + N1*(N2-1-k2)]
      float2 zm;
      if (w == 0) {
        const float2 own0 = v[brev_c((N2 - k2) % N2, N2)];       // k1 = 0: Z[N1*(N2-k2)]
        zm = s ? own1 : own0;
      } else {
        zm = shfl_xor2(own1, 16);                     // partner lane holds k1' = N1 - k1: its Z[k1' + N1*(N2-1-k2)] = Z[N-k]
      }
      if (k2 == N2 / 2 && s != 0) continue;
      const float2 zk = v[j];
      zm.y = -zm.y;                                   // conj(Z[N-k])
      // A = (zk + zm)/2 ; B = -i (zk - zm)/2 ; ortho scale folded into sc
      const float4 o = make_float4((zk.x + zm.x) * sc, (zk.y + zm.y) * sc, (zk.y - zm.y) * sc, -(zk.x - zm.x) * sc);
      const int k = k1 + N1 * k2;
      *reinterpret_cast<float4*>(dst0 + (size_t)k * H * kC) = o;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// P3: rows inverse + fused adds.  grid = ceil(B*H / RPB)
// ------------------------------------------------------------------------------------------------
template <int N1, int N2>
__global__ void __launch_bounds__(kThreadsFft) fft_rows_inv_kernel(const float2* __restrict__ spec, const float* __restrict__ add1,
                                                                 const float* __restrict__ add2, float* __restrict__ out, int H,
                                                                 int nrows) {
  mtd_pdl_prologue();
  using Cfg = RowsCfg<N1, N2>;
  constexpr int N = Cfg::N, Wh = N / 2 + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* T = reinterpret_cast<float2*>(smem_raw);                 // [RPB][k1][n2][q]
  float2* tw = T + (size_t)Cfg::RPB * N * kQ;
  fill_twiddles(tw, N);
  __syncthreads();
  // ---- step A': thread (q, k1) loads its half-spectrum entries, rebuilds Z[k1 + N1*k2] for all k2 (the upper half
  //      comes from the partner lane: Z[N-k] = conj(A_k) + i conj(B_k)), N2-point inverse FFT over k2
  for (int it = threadIdx.x; it < Cfg::RPB * Cfg::IB; it += kThreadsFft) {
    const int r = it / Cfg::IB, rem = it - r * Cfg::IB;
    const int w = rem >> 5, lane = rem & 31, s = lane >> 4, q = lane & 15;
    const long long row = (long long)blockIdx.x * Cfg::RPB + r;
    if (row >= nrows) continue;                       // warp-uniform
    const int k1 = pair_k1<N1>(w, s);
    const int b = (int)(row / H), h = (int)(row - (long long)b * H);
    const float2* src0 = spec + ((size_t)b * Wh * H + h) * kC + 2 * q;
    float2 z[N2];
#pragma unroll
    for (int k2 = 0; k2 < N2 / 2; ++k2) {
      const int k = k1 + N1 * k2;
      const float4 v = __ldg(reinterpret_cast<const float4*>(src0 + (size_t)k * H * kC));   // A = (v.x, v.y), B = (v.z, v.w)
      const float2 zk = make_float2(v.x - v.w, v.y + v.z);          // A + iB
      const float2 zmir = make_float2(v.x + v.w, v.z - v.y);        // conj(A) + i conj(B) = Z[N-k]
      if (w == 0) {
        if (k2 == 0) {
          // k1 = 0: k = 0, imaginary parts dropped (SURVEY A1); k1 = N1/2: an ordinary entry
          z[0] = s ? zk : make_float2(v.x, v.z);
          if (N2 > 1) z[N2 - 1] = zmir;               // only meaningful for k1 = N1/2 (overwritten below for k1 = 0)
        } else {
          z[k2] = zk;
          // k1 = 0: Z[N - N1*k2] lives at k2' = N2 - k2; k1 = N1/2: at k2' = N2 - 1 - k2
          if (s) z[N2 - 1 - k2] = zmir; else z[N2 - k2] = zmir;
        }
      } else {
        z[k2] = zk;
        z[N2 - 1 - k2] = shfl_xor2(zmir, 16);         // partner's mirrored entry is my Z[k1 + N1*(N2-1-k2)]
      }
    }
    if (w == 0) {
      // k1 = 0 also owns k = N/2 (k2 = N2/2), imaginary parts dropped; for k1 = N1/2 every register is already set
      const float4 v = __ldg(reinterpret_cast<const float4*>(src0 + (size_t)(N / 2) * H * kC));
      if (!s) z[N2 / 2] = make_float2(v.x, v.z);
    }
    fft_reg<N2, true>(z);                             // z[j] = u[k1][n2 = brev(j)]
#pragma unroll
    for (int j = 0; j < N2; ++j) {
      const int n2 = brev_c(j, N2);
      const float2 tws = tw[(n2 * k1) & (N - 1)];
      T[((r * N1 + k1) * N2 + n2) * kQ + q] = cmulc(z[j], tws);     // * conj(W_N^(n2 k1))
    }
  }
  __syncthreads();
  // ---- step B': thread (q, n2): N1-point inverse FFT over k1, scale, fused adds, store
  const float sc = rsqrtf((float)N);
  for (int it = threadIdx.x; it < Cfg::RPB * Cfg::IA; it += kThreadsFft) {
    const int r = it / Cfg::IA, rem = it - r * Cfg::IA;
    const int n2 = rem >> 4, q = rem & 15;
    const long long row = (long long)blockIdx.x * Cfg::RPB + r;
    if (row >= nrows) continue;
    float2 v[N1];
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) v[k1] = T[((r * N1 + k1) * N2 + n2) * kQ + q];
    fft_reg<N1, true>(v);                             // v[i] = z[n2 + N2 * brev(i)]
    const size_t base = (size_t)row * N * kC + 2 * q;
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int n = n2 + N2 * brev_c(i, N1);
      const size_t o = base + (size_t)n * kC;
      float2 val = make_float2(v[i].x * sc, v[i].y * sc);
      if (add1) { const float2 t = __ldg(reinterpret_cast<const float2*>(add1 + o)); val.x += t.x; val.y += t.y; }
      if (add2) { const float2 t = __ldg(reinterpret_cast<const float2*>(add2 + o)); val.x += t.x; val.y += t.y; }
      *reinterpret_cast<float2*>(out + o) = val;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// column transforms on a [H][32] complex slice in shared memory; lane = channel.
// forward: global (natural h) -> S in [k1][k2] order;  inverse: S in [k1][k2] order -> global (natural h)
// ------------------------------------------------------------------------------------------------
// RS: row stride of S in float2 (32 = dense; 34 = padded so that the mma fragment loads of the channel mix are conflict-free)
template <int N1, int N2, int RS = kC>
__device__ __forceinline__ void cols_forward(const float2* __restrict__ src, float2* S, const float2* tw) {
  constexpr int N = N1 * N2;
  for (int it = threadIdx.x; it < kC * N2; it += blockDim.x) {          // step A: thread (c, n2)
    const int n2 = it >> 5, c = it & 31;
    float2 v[N1];
#pragma unroll
    for (int n1 = 0; n1 < N1; ++n1) v[n1] = __ldg(src + (size_t)(N2 * n1 + n2) * kC + c);
    fft_reg<N1, false>(v);
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int k1 = brev_c(i, N1);
      S[(k1 * N2 + n2) * RS + c] = k1 == 0 ? v[i] : cmul(v[i], tw[(n2 * k1) & (N - 1)]);
    }
  }
  __syncthreads();
  for (int it = threadIdx.x; it < kC * N1; it += blockDim.x) {          // step B: thread (c, k1), in place
    const int k1 = it >> 5, c = it & 31;
    float2 v[N2];
#pragma unroll
    for (int n2 = 0; n2 < N2; ++n2) v[n2] = S[(k1 * N2 + n2) * RS + c];
    fft_reg<N2, false>(v);
#pragma unroll
    for (int j = 0; j < N2; ++j) S[(k1 * N2 + brev_c(j, N2)) * RS + c] = v[j];     // row k1*N2 + k2 holds X[k1 + N1*k2]
  }
  __syncthreads();
}

template <int N1, int N2, int RS = kC>
__device__ __forceinline__ void cols_inverse(float2* S, const float2* tw, float2* __restrict__ dst, float scale) {
  constexpr int N = N1 * N2;
  for (int it = threadIdx.x; it < kC * N1; it += blockDim.x) {          // step A': thread (c, k1), in place
    const int k1 = it >> 5, c = it & 31;
    float2 v[N2];
#pragma unroll
    for (int k2 = 0; k2 < N2; ++k2) v[k2] = S[(k1 * N2 + k2) * RS + c];
    fft_reg<N2, true>(v);
#pragma unroll
    for (int j = 0; j < N2; ++j) {
      const int n2 = brev_c(j, N2);
      S[(k1 * N2 + n2) * RS + c] = k1 == 0 ? v[j] : cmulc(v[j], tw[(n2 * k1) & (N - 1)]);
    }
  }
  __syncthreads();
  for (int it = threadIdx.x; it < kC * N2; it += blockDim.x) {          // step B': thread (c, n2) -> global
    const int n2 = it >> 5, c = it & 31;
    float2 v[N1];
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) v[k1] = S[(k1 * N2 + n2) * RS + c];
    fft_reg<N1, true>(v);
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int h = n2 + N2 * brev_c(i, N1);
      dst[(size_t)h * kC + c] = make_float2(v[i].x * scale, v[i].y * scale);
    }
  }
}

// ---- channel mix on the tensor cores (legacy warp-level path: mma.sync m16n8k8 TF32, error-compensated 3xTF32) -----------
// A row of S is one frequency: 64 floats [Re c0, Im c0, Re c1, Im c1, ...] = the K index kk (input j = pi(kk) =
// (kk >> 1) + 32 (kk & 1) of the reference's cat[Re, Im] order); the outputs are produced in the same interleaved order.
// Bhi / Blo: [nn][kk] (row stride kMixLd), B[kk][nn] = w[pi(nn)][pi(kk)] / sqrt(H) split into tf32 hi / lo.
// Rows are padded to 68 floats so that the A fragments (rows g, g+8; columns t, t+4) and the B fragments hit 32 banks.
constexpr int kMixLd = 68, kRSmma = kMixLd / 2;
__device__ __forceinline__ int mix_pi(int kk) { return (kk >> 1) + 32 * (kk & 1); }
__device__ __forceinline__ uint32_t tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mix_prepare(const float* __restrict__ w, const float* __restrict__ bias, float scale, float* Bhi,
                                            float* Blo, float* bsI) {
  for (int i = threadIdx.x; i < kC2 * kC2; i += blockDim.x) {
    const int nn = i >> 6, kk = i & 63;
    const float v = __ldg(w + mix_pi(nn) * kC2 + mix_pi(kk)) * scale;
    const uint32_t h = tf32_rna(v);
    Bhi[nn * kMixLd + kk] = __uint_as_float(h);
    Blo[nn * kMixLd + kk] = __uint_as_float(tf32_rna(v - __uint_as_float(h)));
  }
  if (threadIdx.x < kC2) bsI[threadIdx.x] = __ldg(bias + mix_pi(threadIdx.x));
}

// Bt[kk][nn] = w[pi(nn)][pi(kk)] (transposed, unscaled): the B operand of dy = gz W in the backward kernel
__device__ __forceinline__ void mix_prepare_t(const float* __restrict__ w, float* Bhi, float* Blo) {
  for (int i = threadIdx.x; i < kC2 * kC2; i += blockDim.x) {
    const int kk = i >> 6, nn = i & 63;
    const float v = __ldg(w + mix_pi(nn) * kC2 + mix_pi(kk));
    const uint32_t h = tf32_rna(v);
    Bhi[kk * kMixLd + nn] = __uint_as_float(h);
    Blo[kk * kMixLd + nn] = __uint_as_float(tf32_rna(v - __uint_as_float(h)));
  }
}

// out[r][nn] = relu( bias + sum_kk S[r][kk] B[kk][nn] ), in place on the padded rows of S.  Work item = (16-row block, NT/8
// of the 8 column tiles); a warp's items are processed in rounds with a block barrier between compute and store when two
// warps share rows (H = 64), so no warp overwrites a row another warp still reads.
// MODE 0: Out = relu(bias + A B), Out may alias A (forward mix);  MODE 1: Out[r][n] = 0 where !(bias + A B > 0)
// (ReLU mask of the recomputed pre-activation applied to the gradient rows);  MODE 2: Out = A B (no bias).
template <int H, int THREADS, int MODE>
__device__ __forceinline__ void mix_mma(const float2* A, float2* Out, const float* Bhi, const float* Blo, const float* bsI) {
  constexpr int NW = THREADS / 32, RB = H / 16;
  constexpr int NSPLIT = RB >= NW ? 1 : NW / RB;           // column split when there are fewer row blocks than warps
  constexpr int NT = 8 / NSPLIT;                           // 8-column tiles per item
  constexpr int ITEMS = RB * NSPLIT, ROUNDS = (ITEMS + NW - 1) / NW;
  static_assert(NSPLIT == 1 || NSPLIT == 2 || NSPLIT == 4, "column split");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* Sf = reinterpret_cast<const float*>(A);
  float* Of = reinterpret_cast<float*>(Out);
#pragma unroll 1
  for (int round = 0; round < ROUNDS; ++round) {
    const int item = round * NW + warp;
    const bool active = item < ITEMS;
    const int rb = active ? item / NSPLIT : 0, n0 = (item % NSPLIT) * NT;
    float acc[NT][4], acc2[NT][4];
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      const float b0 = MODE == 2 ? 0.f : bsI[(n0 + n) * 8 + 2 * t], b1 = MODE == 2 ? 0.f : bsI[(n0 + n) * 8 + 2 * t + 1];
      acc[n][0] = b0; acc[n][1] = b1; acc[n][2] = b0; acc[n][3] = b1;
      acc2[n][0] = acc2[n][1] = acc2[n][2] = acc2[n][3] = 0.f;
    }
    const float* r0 = Sf + (size_t)(rb * 16 + g) * kMixLd;
    const float* r1 = r0 + 8 * kMixLd;
    if (active) {
#pragma unroll 2
      for (int k0 = 0; k0 < kC2; k0 += 8) {
        const float av[4] = {r0[k0 + t], r1[k0 + t], r0[k0 + t + 4], r1[k0 + t + 4]};
        uint32_t ah[4], al[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          ah[i] = tf32_rna(av[i]);
          al[i] = tf32_rna(av[i] - __uint_as_float(ah[i]));
        }
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          const float* bh = Bhi + ((n0 + n) * 8 + g) * kMixLd + k0 + t;
          const float* bl = Blo + ((n0 + n) * 8 + g) * kMixLd + k0 + t;
          const uint32_t bh0 = __float_as_uint(bh[0]), bh1 = __float_as_uint(bh[4]);
          const uint32_t bl0 = __float_as_uint(bl[0]), bl1 = __float_as_uint(bl[4]);
          mma_tf32(acc2[n], al, bh0, bh1);
          mma_tf32(acc2[n], ah, bl0, bl1);
          mma_tf32(acc[n], ah, bh0, bh1);
        }
      }
    }
    if (MODE == 0) { if (NSPLIT > 1) __syncthreads(); else __syncwarp(); }      // in place: all reads of these rows are done
    if (active) {
      float* w0 = Of + (size_t)(rb * 16 + g) * kMixLd;
      float* w1 = w0 + 8 * kMixLd;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        const int col = (n0 + n) * 8 + 2 * t;
        const float v0 = acc[n][0] + acc2[n][0], v1 = acc[n][1] + acc2[n][1], v2 = acc[n][2] + acc2[n][2], v3 = acc[n][3] + acc2[n][3];
        if (MODE == 0) {
          *reinterpret_cast<float2*>(w0 + col) = make_float2(fmaxf(v0, 0.f), fmaxf(v1, 0.f));
          *reinterpret_cast<float2*>(w1 + col) = make_float2(fmaxf(v2, 0.f), fmaxf(v3, 0.f));
        } else if (MODE == 1) {
          if (!(v0 > 0.f)) w0[col] = 0.f;
          if (!(v1 > 0.f)) w0[col + 1] = 0.f;
          if (!(v2 > 0.f)) w1[col] = 0.f;
          if (!(v3 > 0.f)) w1[col + 1] = 0.f;
        } else {
          *reinterpret_cast<float2*>(w0 + col) = make_float2(v0, v1);
          *reinterpret_cast<float2*>(w1 + col) = make_float2(v2, v3);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// P2: columns + channel mix.  grid = B*Wh.   smem: S[H][32] float2 | Mt[64][64] | bias[64] | tw[H]
// ------------------------------------------------------------------------------------------------
// THREADS: 256 for H <= 128; 512 for the 256- / 512-point columns, where one CTA owns the SM (128 KB slice) and the
// transform phases are latency-bound on too few warps otherwise
template <int N1, int N2, int THREADS>
__global__ void __launch_bounds__(THREADS) fft_cols_mix_kernel(const float2* __restrict__ spec_in, float2* __restrict__ spec_out,
                                                             const float* __restrict__ w, const float* __restrict__ bias) {
  mtd_pdl_prologue();
  constexpr int H = N1 * N2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* S = reinterpret_cast<float2*>(smem_raw);                   // [H][kRSmma] (rows padded to 68 floats)
  float* Bhi = reinterpret_cast<float*>(S + (size_t)H * kRSmma);     // [64][68] tf32 hi of w[pi(nn)][pi(kk)] / sqrt(H)
  float* Blo = Bhi + kC2 * kMixLd;
  float* bs = Blo + kC2 * kMixLd;                                    // bias in interleaved output order
  float2* tw = reinterpret_cast<float2*>(bs + kC2);
  const size_t slice = (size_t)blockIdx.x * H * kC;
  const float sH = rsqrtf((float)H);
  fill_twiddles(tw, H);
  mix_prepare(w, bias, sH, Bhi, Blo, bs);
  __syncthreads();
  cols_forward<N1, N2, kRSmma>(spec_in + slice, S, tw);
  mix_mma<H, THREADS, 0>(S, S, Bhi, Blo, bs);
  __syncthreads();
  cols_inverse<N1, N2, kRSmma>(S, tw, spec_out + slice, sH);
}

// ------------------------------------------------------------------------------------------------
// Backward of P2.  grid = B*Wh
// smem: S[H][32] | T[H][32] | Mt[64][64] | Mn[64][64] | bias[64] | tw[H]
// part: per CTA 64*64 dW partial followed by 64 db partial
// ------------------------------------------------------------------------------------------------
template <int N1, int N2>
__global__ void __launch_bounds__(kThreadsFft) fft_cols_mix_bwd_kernel(const float2* __restrict__ spec_x, const float2* __restrict__ spec_g,
                                                                     float2* __restrict__ spec_out, const float* __restrict__ w,
                                                                     const float* __restrict__ bias, float* __restrict__ part,
                                                                     const float* __restrict__ bw, int Wh, int W) {
  mtd_pdl_prologue();
  constexpr int H = N1 * N2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* S = reinterpret_cast<float2*>(smem_raw);                   // [H][kRSmma]
  float2* T = S + (size_t)H * kRSmma;
  float* bs = reinterpret_cast<float*>(T + (size_t)H * kRSmma);
  float2* tw = reinterpret_cast<float2*>(bs + kC2);
  // tf32 hi / lo mix operands, prepared once per call by fft_mix_prepare_kernel (L1 / L2 resident, shared by all CTAs):
  // forward operand (scaled by 1/sqrt(H)) and the transposed, unscaled one for dy = gz W
  const float* Bhi = bw;
  const float* Blo = Bhi + kC2 * kMixLd;
  const float* Thi = Blo + kC2 * kMixLd;
  const float* Tlo = Thi + kC2 * kMixLd;
  const size_t slice = (size_t)blockIdx.x * H * kC;
  const int kw = blockIdx.x % Wh;
  const float wk = (kw == 0 || kw == (W >> 1)) ? 1.f : 2.f;
  const float sH = rsqrtf((float)H);
  fill_twiddles(tw, H);
  if (threadIdx.x < kC2) bs[threadIdx.x] = __ldg(bias + mix_pi(threadIdx.x));
  __syncthreads();
  cols_forward<N1, N2, kRSmma>(spec_x + slice, S, tw);        // S = FFT_H(X1) (unscaled), rows in [k1][k2] order
  cols_forward<N1, N2, kRSmma>(spec_g + slice, T, tw);        // T = FFT_H(G)  -- same row order, so masks / products line up

  // 1) ReLU mask from the recomputed pre-activation; gz = mask * G2 (left unscaled) written in place (tensor cores)
  mix_mma<H, kThreadsFft, 1>(S, T, Bhi, Blo, bs);
  __syncthreads();
  // 2) dW / db partials: dW[o][j] = wk/H * sum_r gz[r][o] * y[r][j]; db[o] = wk/sqrt(H) * sum_r gz[r][o]
  //    on the tensor cores: D[nn][kk] = sum_r T[r][nn] S[r][kk] in the interleaved index space (both operands are data:
  //    both are split into tf32 hi / lo); warp w owns output rows 16 (w >> 1) .. +15 and columns 32 (w & 1) .. +31
  {
    const float* Tf = reinterpret_cast<const float*>(T);
    const float* Sf = reinterpret_cast<const float*>(S);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const int m0 = (warp >> 1) * 16, nb = (warp & 1) * 32;
    float acc[4][4], acc2[4][4];
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[n][e] = acc2[n][e] = 0.f;
#pragma unroll 2
    for (int k0 = 0; k0 < H; k0 += 8) {
      const float* ta = Tf + (size_t)(k0 + t) * kMixLd + m0 + g;
      const float av[4] = {ta[0], ta[8], ta[4 * kMixLd], ta[4 * kMixLd + 8]};      // (m, k) = (g, t), (g+8, t), (g, t+4), (g+8, t+4)
      uint32_t ah[4], al[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        ah[i] = tf32_rna(av[i]);
        al[i] = tf32_rna(av[i] - __uint_as_float(ah[i]));
      }
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const float* sb = Sf + (size_t)(k0 + t) * kMixLd + nb + n * 8 + g;         // (k, n) = (t, g), (t+4, g)
        const float b0 = sb[0], b1 = sb[4 * kMixLd];
        const uint32_t bh0 = tf32_rna(b0), bh1 = tf32_rna(b1);
        const uint32_t bl0 = tf32_rna(b0 - __uint_as_float(bh0)), bl1 = tf32_rna(b1 - __uint_as_float(bh1));
        mma_tf32(acc2[n], al, bh0, bh1);
        mma_tf32(acc2[n], ah, bl0, bl1);
        mma_tf32(acc[n], ah, bh0, bh1);
      }
    }
    float* p = part + (size_t)blockIdx.x * (kC2 * kC2 + kC2);
    const float sW = wk * sH * sH;
    const int o0 = mix_pi(m0 + g), o1 = mix_pi(m0 + g + 8);
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      const int j0 = mix_pi(nb + n * 8 + 2 * t), j1 = mix_pi(nb + n * 8 + 2 * t + 1);
      p[o0 * kC2 + j0] = (acc[n][0] + acc2[n][0]) * sW;
      p[o0 * kC2 + j1] = (acc[n][1] + acc2[n][1]) * sW;
      p[o1 * kC2 + j0] = (acc[n][2] + acc2[n][2]) * sW;
      p[o1 * kC2 + j1] = (acc[n][3] + acc2[n][3]) * sW;
    }
    if (threadIdx.x < kC2) {                                     // db: column sums of gz
      float sum = 0.f;
      for (int r = 0; r < H; ++r) sum += Tf[(size_t)r * kMixLd + threadIdx.x];
      p[kC2 * kC2 + mix_pi(threadIdx.x)] = sum * wk * sH;
    }
  }
  __syncthreads();
  // 3) dy[r][j] = sum_o gz[r][o] * w[o][j]   (unscaled; 1/H applied at the store)  -> S (tensor cores)
  mix_mma<H, kThreadsFft, 2>(T, S, Thi, Tlo, nullptr);
  __syncthreads();
  cols_inverse<N1, N2, kRSmma>(S, tw, spec_out + slice, sH * sH);
}

// one block: the four tf32 operand matrices of the backward kernel's tensor-core phases -> bw[4][64][kMixLd]
__global__ void __launch_bounds__(256) fft_mix_prepare_kernel(const float* __restrict__ w, float scale, float* __restrict__ bw) {
  mtd_pdl_prologue();
  float* Bhi = bw;
  float* Blo = Bhi + kC2 * kMixLd;
  for (int i = threadIdx.x; i < kC2 * kC2; i += blockDim.x) {
    const int nn = i >> 6, kk = i & 63;
    const float v = __ldg(w + mix_pi(nn) * kC2 + mix_pi(kk)) * scale;
    const uint32_t h = tf32_rna(v);
    Bhi[nn * kMixLd + kk] = __uint_as_float(h);
    Blo[nn * kMixLd + kk] = __uint_as_float(tf32_rna(v - __uint_as_float(h)));
  }
  mix_prepare_t(w, Blo + kC2 * kMixLd, Blo + 2 * kC2 * kMixLd);
}

// dW / db = ordered sum of the per-CTA partials.  32 output elements per block, 8 lanes of partial index per element:
// lane g sums partials p = g, g + 8, ... (Kahan), the eight lane sums are added in lane order -- deterministic, and 8 x
// the parallelism of one thread per element (660 partials of 16.6 KB at B = 20).
__global__ void __launch_bounds__(256) fft_wgrad_reduce_kernel(const float* __restrict__ part, int nparts, float* __restrict__ dw,
                                                              float* __restrict__ db) {
  mtd_pdl_prologue();
  __shared__ float sh[8][33];
  const int per = kC2 * kC2 + kC2;
  const int e = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + e;
  float s = 0.f, comp = 0.f;     // Kahan: hundreds of partials of mixed sign
  if (i < per) {
    for (int p = g; p < nparts; p += 8) {
      const float v = __ldg(part + (size_t)p * per + i) - comp;
      const float t = s + v;
      comp = (t - s) - v;
      s = t;
    }
  }
  sh[g][e] = s;
  __syncthreads();
  if (g == 0 && i < per) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += sh[k][e];
    if (i < kC2 * kC2) dw[i] = tot;
    else db[i - kC2 * kC2] = tot;
  }
}

// ------------------------------------------------------------------------------------------------
// Bluestein (chirp-z) transforms for every other length N <= 512:
//   X[k] = c[k] sum_n (x[n] c[n]) conj(c[k - n]),   c[n] = exp(-i pi n^2 / N)
// The convolution runs circularly at M = max(64, pow2 >= 2N - 1) <= 1024 on the four-step transforms above:
//   step A   thread (n2, l): x[n] c[n] at n = N2*n1 + n2 (0 for n >= N), N1-point FFT, twiddle -> S[k1][n2]
//   step BA  thread (k1, l): N2-point FFT, * Bh[k1 + N1*k2], N2-point inverse FFT, conj twiddle -> S[k1][n2] in place
//            (the pointwise product is frequency-local, so the forward and the inverse transform meet in registers)
//   step B'  thread (n2, l): N1-point inverse FFT, * c[n] -> store(n, l, .) for n < N, after a barrier (S is free)
// Bh = FFT_M(conj(c) wrapped circularly) / M.  INV (the unnormalised inverse DFT) uses conj(c) and conj(Bh): the wrapped
// chirp is symmetric, so FFT_M of its conjugate is conj(Bh).
// kNL = 16 interleaved complex sequences per CTA: the 16 channel pairs of one image row, or 16 channels of one (b, kw)
// column slice.  S[M][16] is 128 KB at M = 1024.
// ------------------------------------------------------------------------------------------------
constexpr int kNL = 16;

template <int N1, int N2>
struct BlueCfg {
  static constexpr int M = N1 * N2;
  static constexpr int THREADS = (N1 > N2 ? N1 : N2) * kNL;          // at most one item per thread in every step
  static constexpr size_t smem = (size_t)M * kNL * 8 + (size_t)M * 8;   // S | tw
};

template <int N1, int N2, bool INV, class Load, class Store>
__device__ __forceinline__ void bluestein(float2* S, float2* tw, const float2* __restrict__ chirp, const float2* __restrict__ bh,
                                          int N, Load load, Store store) {
  constexpr int M = N1 * N2;
  const int l = threadIdx.x & (kNL - 1), t = threadIdx.x / kNL;
  fill_twiddles(tw, M);
  __syncthreads();
  if (t < N2) {                                                        // step A
    const int n2 = t;
    float2 v[N1];
#pragma unroll
    for (int n1 = 0; n1 < N1; ++n1) {
      const int n = N2 * n1 + n2;
      v[n1] = make_float2(0.f, 0.f);
      if (n < N) {
        const float2 x = load(n, l), c = __ldg(chirp + n);
        v[n1] = INV ? cmulc(x, c) : cmul(x, c);
      }
    }
    fft_reg<N1, false>(v);
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int k1 = brev_c(i, N1);
      S[(k1 * N2 + n2) * kNL + l] = k1 == 0 ? v[i] : cmul(v[i], tw[(n2 * k1) & (M - 1)]);
    }
  }
  __syncthreads();
  if (t < N1) {                                                        // step BA
    const int k1 = t;
    float2 v[N2], z[N2];
#pragma unroll
    for (int n2 = 0; n2 < N2; ++n2) v[n2] = S[(k1 * N2 + n2) * kNL + l];
    fft_reg<N2, false>(v);                                             // v[j] = Y[k1 + N1 * brev(j)]
#pragma unroll
    for (int j = 0; j < N2; ++j) {
      const int k2 = brev_c(j, N2);
      const float2 b = __ldg(bh + k1 + N1 * k2);
      z[k2] = INV ? cmulc(v[j], b) : cmul(v[j], b);
    }
    fft_reg<N2, true>(z);                                              // z[j] = y[k1][n2 = brev(j)]
#pragma unroll
    for (int j = 0; j < N2; ++j) {
      const int n2 = brev_c(j, N2);
      S[(k1 * N2 + n2) * kNL + l] = k1 == 0 ? z[j] : cmulc(z[j], tw[(n2 * k1) & (M - 1)]);
    }
  }
  __syncthreads();
  float2 v[N1];                                                        // step B'
  const int n2 = t;
  if (t < N2) {
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) v[k1] = S[(k1 * N2 + n2) * kNL + l];
    fft_reg<N1, true>(v);                                              // v[i] = y[n2 + N2 * brev(i)]
  }
  __syncthreads();
  if (t < N2) {
#pragma unroll
    for (int i = 0; i < N1; ++i) {
      const int n = n2 + N2 * brev_c(i, N1);
      if (n < N) {
        const float2 c = __ldg(chirp + n);
        store(n, l, INV ? cmulc(v[i], c) : cmul(v[i], c));
      }
    }
  }
}

// P1 at any W: one image row per CTA.  grid = B*H
template <int N1, int N2>
__global__ void __launch_bounds__(BlueCfg<N1, N2>::THREADS) fft_rows_fwd_blue_kernel(const float* __restrict__ x, float2* __restrict__ spec,
                                                                                    int H, int W, const float2* __restrict__ chirp,
                                                                                    const float2* __restrict__ bh) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* S = reinterpret_cast<float2*>(smem_raw);                     // [M][16]; Z[k][q] after the transform
  float2* tw = S + (size_t)N1 * N2 * kNL;
  const long long row = blockIdx.x;
  const float2* src = reinterpret_cast<const float2*>(x + (size_t)row * W * kC);     // src[n * 16 + q] = (x_2q, x_2q+1)[n]
  bluestein<N1, N2, false>(S, tw, chirp, bh, W, [&](int n, int q) { return __ldg(src + (size_t)n * kQ + q); },
                           [&](int k, int q, float2 z) { S[k * kNL + q] = z; });
  __syncthreads();
  // real-pair separation A_k = (Z_k + conj Z_{W-k}) / 2, B_k = -i (Z_k - conj Z_{W-k}) / 2 for k <= W/2
  const int Wh = W / 2 + 1, b = (int)(row / H), h = (int)(row - (long long)b * H);
  float2* dst0 = spec + ((size_t)b * Wh * H + h) * kC;
  const float sc = rsqrtf((float)W) * 0.5f;
  for (int i = threadIdx.x; i < Wh * kQ; i += blockDim.x) {
    const int k = i / kQ, q = i % kQ;
    const float2 zk = S[k * kNL + q];
    float2 zm = S[(k == 0 ? 0 : W - k) * kNL + q];
    zm.y = -zm.y;
    const float4 o = make_float4((zk.x + zm.x) * sc, (zk.y + zm.y) * sc, (zk.y - zm.y) * sc, -(zk.x - zm.x) * sc);
    *reinterpret_cast<float4*>(dst0 + (size_t)k * H * kC + 2 * q) = o;
  }
}

// P3 at any W: one image row per CTA, fused residual adds.  grid = B*H.  The imaginary parts of kw = 0, and of kw = W/2
// when W is even, are dropped (SURVEY A1); an odd W has no Nyquist column.
template <int N1, int N2>
__global__ void __launch_bounds__(BlueCfg<N1, N2>::THREADS) fft_rows_inv_blue_kernel(const float2* __restrict__ spec,
                                                                                    const float* __restrict__ add1,
                                                                                    const float* __restrict__ add2,
                                                                                    float* __restrict__ out, int H, int W,
                                                                                    const float2* __restrict__ chirp,
                                                                                    const float2* __restrict__ bh) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* S = reinterpret_cast<float2*>(smem_raw);
  float2* tw = S + (size_t)N1 * N2 * kNL;
  const long long row = blockIdx.x;
  const int Wh = W / 2 + 1, b = (int)(row / H), h = (int)(row - (long long)b * H);
  const float2* src0 = spec + ((size_t)b * Wh * H + h) * kC;
  const float sc = rsqrtf((float)W);
  const size_t base = (size_t)row * W * kC;
  bluestein<N1, N2, true>(
      S, tw, chirp, bh, W,
      [&](int n, int q) {                                              // Z[n] = A_n + i B_n;  Z[W-n] = conj(A_n) + i conj(B_n)
        const bool up = n >= Wh;
        const float4 v = __ldg(reinterpret_cast<const float4*>(src0 + (size_t)(up ? W - n : n) * H * kC + 2 * q));
        if (n == 0 || 2 * n == W) return make_float2(v.x, v.z);
        return up ? make_float2(v.x + v.w, v.z - v.y) : make_float2(v.x - v.w, v.y + v.z);
      },
      [&](int n, int q, float2 z) {
        const size_t o = base + (size_t)n * kC + 2 * q;
        float2 val = make_float2(z.x * sc, z.y * sc);
        if (add1) { const float2 a = __ldg(reinterpret_cast<const float2*>(add1 + o)); val.x += a.x; val.y += a.y; }
        if (add2) { const float2 a = __ldg(reinterpret_cast<const float2*>(add2 + o)); val.x += a.x; val.y += a.y; }
        *reinterpret_cast<float2*>(out + o) = val;
      });
}

// P2 at any H, column transform of 16 channels of one (b, kw) slice: out = scale * DFT_H(in) (INV: inverse DFT).
// grid = 2 * B*Wh.  May run in place (in == out): a CTA reads its columns before it writes them.
template <int N1, int N2, bool INV>
__global__ void __launch_bounds__(BlueCfg<N1, N2>::THREADS) fft_cols_blue_kernel(const float2* in, float2* out, int H, float scale,
                                                                                const float2* __restrict__ chirp,
                                                                                const float2* __restrict__ bh) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* S = reinterpret_cast<float2*>(smem_raw);
  float2* tw = S + (size_t)N1 * N2 * kNL;
  const size_t off = (size_t)(blockIdx.x >> 1) * H * kC + (blockIdx.x & 1) * kNL;
  const float2* src = in + off;
  float2* dst = out + off;
  bluestein<N1, N2, INV>(S, tw, chirp, bh, H, [&](int n, int c) { return src[(size_t)n * kC + c]; },
                         [&](int k, int c, float2 z) { dst[(size_t)k * kC + c] = make_float2(z.x * scale, z.y * scale); });
}

// P2 at any H, channel mix: every row of the spectrum is one frequency, mixed independently (in place):
// row = relu(bias + row M), M = w / sqrt(H) in the interleaved index space.  128 rows per CTA.  grid = ceil(nrows / 128)
constexpr int kMixRows = 128, kThreadsMix = 256;
__global__ void __launch_bounds__(kThreadsMix) fft_mix_rows_kernel(float2* spec, const float* __restrict__ w, const float* __restrict__ bias,
                                                                  long long nrows, float scale) {
  mtd_pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Sf = reinterpret_cast<float*>(smem_raw);                      // [128][kMixLd]
  float* Bhi = Sf + kMixRows * kMixLd;
  float* Blo = Bhi + kC2 * kMixLd;
  float* bs = Blo + kC2 * kMixLd;
  mix_prepare(w, bias, scale, Bhi, Blo, bs);
  const long long r0 = (long long)blockIdx.x * kMixRows;
  float4* g = reinterpret_cast<float4*>(spec) + r0 * (kC2 / 4);
  for (int i = threadIdx.x; i < kMixRows * (kC2 / 4); i += kThreadsMix) {
    const int r = i / (kC2 / 4), c = i % (kC2 / 4);
    *reinterpret_cast<float4*>(Sf + r * kMixLd + 4 * c) = r0 + r < nrows ? g[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  mix_mma<kMixRows, kThreadsMix, 0>(reinterpret_cast<float2*>(Sf), reinterpret_cast<float2*>(Sf), Bhi, Blo, bs);
  __syncthreads();
  for (int i = threadIdx.x; i < kMixRows * (kC2 / 4); i += kThreadsMix) {
    const int r = i / (kC2 / 4), c = i % (kC2 / 4);
    if (r0 + r < nrows) g[i] = *reinterpret_cast<const float4*>(Sf + r * kMixLd + 4 * c);
  }
}

int blue_len(int n) {
  int m = 64;
  while (m < 2 * n - 1) m <<= 1;
  return m;
}

// chirp c[n] (n < N) and Bh[k] (k < M) of a length, built once per (device, length) on the host in fp64 and kept on the
// device for the life of the process (12 KB at most per length).  The phase pi n^2 / N is reduced as n^2 mod 2N in integer
// arithmetic first: formed in fp32, it loses the phase at N ~ 500.
struct BlueTables {
  std::once_flag once;
  int rc = MTD_OK;
  float2* chirp = nullptr;
  float2* bh = nullptr;
};
constexpr int kBlueMaxDev = 16;

int blue_tables(int N, const float2** chirp, const float2** bh) {
  static BlueTables tabs[kBlueMaxDev][513];
  int dev = 0;
  MTD_CUDA(cudaGetDevice(&dev));
  if (dev >= kBlueMaxDev || N < 1 || N > 512) return MTD_EINVAL;
  BlueTables& t = tabs[dev][N];
  std::call_once(t.once, [&] {
    const int M = blue_len(N);
    std::vector<double> cr(M), ci(M), er(M), ei(M);            // cr + i ci: wrapped conj(c);  er + i ei = exp(-2 pi i j / M)
    for (int j = 0; j < M; ++j) {
      er[j] = std::cos(2.0 * M_PI * j / M);
      ei[j] = -std::sin(2.0 * M_PI * j / M);
    }
    std::vector<float2> hc(N), hb(M);
    for (int n = 0; n < N; ++n) {
      const double a = M_PI * (double)(((long long)n * n) % (2LL * N)) / N;
      hc[n] = make_float2((float)std::cos(a), (float)-std::sin(a));
      cr[n] = std::cos(a);
      ci[n] = std::sin(a);
      if (n) { cr[M - n] = cr[n]; ci[M - n] = ci[n]; }
    }
    for (int k = 0; k < M; ++k) {
      double sr = 0.0, si = 0.0;
      for (int m = 0; m < M; ++m) {
        if (m >= N && m <= M - N) continue;                    // the zero padding
        const int j = (int)(((long long)m * k) % M);
        sr += cr[m] * er[j] - ci[m] * ei[j];
        si += cr[m] * ei[j] + ci[m] * er[j];
      }
      hb[k] = make_float2((float)(sr / M), (float)(si / M));
    }
    float2 *dc = nullptr, *db = nullptr;
    cudaError_t e = cudaMalloc(&dc, sizeof(float2) * N);
    if (e == cudaSuccess) e = cudaMalloc(&db, sizeof(float2) * M);
    if (e == cudaSuccess) e = cudaMemcpy(dc, hc.data(), sizeof(float2) * N, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, hb.data(), sizeof(float2) * M, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();        // the copies complete before any stream can read them
    t.rc = (int)e;
    t.chirp = dc;
    t.bh = db;
  });
  *chirp = t.chirp;
  *bh = t.bh;
  return t.rc;
}

// dispatch on the Bluestein convolution length M = N1 x N2
#define MTD_BLUE_DISPATCH(M, CALL)      \
  switch (M) {                          \
    case 64: { CALL(8, 8); break; }     \
    case 128: { CALL(8, 16); break; }   \
    case 256: { CALL(16, 16); break; }  \
    case 512: { CALL(16, 32); break; }  \
    case 1024: { CALL(32, 32); break; } \
    default: return MTD_EINVAL;         \
  }

template <typename K>
int set_smem(K kernel, size_t bytes) {
  if (bytes > 227 * 1024) return MTD_EINVAL;
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
  }
  return MTD_OK;
}

bool fft_len_ok(int n) { return n == 64 || n == 128 || n == 256 || n == 512; }

// dispatch on the transform length: 64 = 8x8, 128 = 8x16, 256 = 16x16, 512 = 16x32
#define MTD_FFT_DISPATCH(LEN, CALL) \
  switch (LEN) {                    \
    case 64: { CALL(8, 8); break; }   \
    case 128: { CALL(8, 16); break; } \
    case 256: { CALL(16, 16); break; } \
    case 512: { CALL(16, 32); break; } \
    default: return MTD_EINVAL;       \
  }

// P2 column transforms at any H: out = scale * DFT_H(in) (INV: the inverse DFT) over every (b, kw) slice
template <bool INV>
int launch_cols_blue(const float2* in, float2* out, int nslices, int H, float scale, const float2* chirp, const float2* bh,
                     cudaStream_t st) {
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    using Cfg = BlueCfg<N1_, N2_>;                                                                                  \
    int rc = set_smem(fft_cols_blue_kernel<N1_, N2_, INV>, Cfg::smem);                                              \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_cols_blue_kernel<N1_, N2_, INV>, 2 * nslices, Cfg::THREADS, Cfg::smem, st, in, out, H, scale,    \
               chirp, bh);                                                                                          \
  }
  MTD_BLUE_DISPATCH(blue_len(H), CALL)
#undef CALL
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

}  // namespace

extern "C" {

long long mtd_fft_spec_elems(int B, int H, int W, int C) { return (long long)B * (W / 2 + 1) * H * C * 2; }

// per-CTA dW / db partials followed by the four tf32 mix operands of the backward kernel
long long mtd_fft_bwd_part_elems(int B, int W) { return (long long)B * (W / 2 + 1) * (kC2 * kC2 + kC2) + 4LL * kC2 * kMixLd; }

/* 1 when (H, W, C) is a geometry the frequency branch supports: C == 32, 1 <= H, W <= 512. */
int mtd_fft_supported(int H, int W, int C) { return (C == kC && H >= 1 && H <= 512 && W >= 1 && W <= 512) ? 1 : 0; }

int mtd_fft_rows_fwd(const float* x, float* spec, int B, int H, int W, int C, void* stream) {
  MTD_REQUIRE(x && spec && B > 0 && H > 0 && W >= 1 && W <= 512 && C == kC);
  MTD_REQUIRE(mtd_aligned16(x) && mtd_aligned16(spec));
  const int nrows = B * H;
  if (!fft_len_ok(W)) {
    const float2 *chirp, *bh;
    int rc = blue_tables(W, &chirp, &bh);
    if (rc) return rc;
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    using Cfg = BlueCfg<N1_, N2_>;                                                                                  \
    rc = set_smem(fft_rows_fwd_blue_kernel<N1_, N2_>, Cfg::smem);                                                   \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_rows_fwd_blue_kernel<N1_, N2_>, nrows, Cfg::THREADS, Cfg::smem, (cudaStream_t)stream, x,         \
               reinterpret_cast<float2*>(spec), H, W, chirp, bh);                                                   \
  }
    MTD_BLUE_DISPATCH(blue_len(W), CALL)
#undef CALL
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    using Cfg = RowsCfg<N1_, N2_>;                                                                                  \
    int rc = set_smem(fft_rows_fwd_kernel<N1_, N2_>, Cfg::smem);                                                    \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_rows_fwd_kernel<N1_, N2_>, (nrows + Cfg::RPB - 1) / Cfg::RPB, kThreadsFft, Cfg::smem, (cudaStream_t)stream, x, \
               reinterpret_cast<float2*>(spec), H, nrows);                                                          \
  }
  MTD_FFT_DISPATCH(W, CALL)
#undef CALL
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int mtd_fft_rows_inv(const float* spec, const float* add1, const float* add2, float* out, int B, int H, int W, int C,
                     void* stream) {
  MTD_REQUIRE(spec && out && B > 0 && H > 0 && W >= 1 && W <= 512 && C == kC);
  MTD_REQUIRE(mtd_aligned16(spec) && mtd_aligned16(out) && mtd_aligned16(add1) && mtd_aligned16(add2));
  const int nrows = B * H;
  if (!fft_len_ok(W)) {
    const float2 *chirp, *bh;
    int rc = blue_tables(W, &chirp, &bh);
    if (rc) return rc;
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    using Cfg = BlueCfg<N1_, N2_>;                                                                                  \
    rc = set_smem(fft_rows_inv_blue_kernel<N1_, N2_>, Cfg::smem);                                                   \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_rows_inv_blue_kernel<N1_, N2_>, nrows, Cfg::THREADS, Cfg::smem, (cudaStream_t)stream,            \
               reinterpret_cast<const float2*>(spec), add1, add2, out, H, W, chirp, bh);                           \
  }
    MTD_BLUE_DISPATCH(blue_len(W), CALL)
#undef CALL
    MTD_CHECK_LAUNCH();
    return MTD_OK;
  }
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    using Cfg = RowsCfg<N1_, N2_>;                                                                                  \
    int rc = set_smem(fft_rows_inv_kernel<N1_, N2_>, Cfg::smem);                                                    \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_rows_inv_kernel<N1_, N2_>, (nrows + Cfg::RPB - 1) / Cfg::RPB, kThreadsFft, Cfg::smem, (cudaStream_t)stream,    \
               reinterpret_cast<const float2*>(spec), add1, add2, out, H, nrows);                                   \
  }
  MTD_FFT_DISPATCH(W, CALL)
#undef CALL
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int mtd_fft_cols_mix(const float* spec_in, float* spec_out, const float* w, const float* bias, int B, int H, int W,
                     int C, void* stream) {
  MTD_REQUIRE(spec_in && spec_out && w && bias && B > 0 && H >= 1 && H <= 512 && W >= 1 && W <= 512 && C == kC);
  MTD_REQUIRE(mtd_aligned16(spec_in) && mtd_aligned16(spec_out));
  if (!fft_len_ok(H)) {
    // column transform, flat channel mix, inverse column transform: a 32-channel M-row slice does not fit in shared
    // memory at M = 1024, so the transforms run on 16-channel halves and the mix on the spectrum in global memory (L2)
    const float2 *chirp, *bh;
    int rc = blue_tables(H, &chirp, &bh);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int nslices = B * (W / 2 + 1);
    const float sH = 1.0f / sqrtf((float)H);
    rc = launch_cols_blue<false>(reinterpret_cast<const float2*>(spec_in), reinterpret_cast<float2*>(spec_out), nslices, H,
                                 1.0f, chirp, bh, st);
    if (rc) return rc;
    const size_t msmem = ((size_t)kMixRows * kMixLd + 2 * kC2 * kMixLd + kC2) * 4;
    rc = set_smem(fft_mix_rows_kernel, msmem);
    if (rc) return rc;
    const long long nrows = (long long)nslices * H;
    mtd_launch(fft_mix_rows_kernel, (unsigned)((nrows + kMixRows - 1) / kMixRows), kThreadsMix, msmem, st,
               reinterpret_cast<float2*>(spec_out), w, bias, nrows, sH);
    MTD_CHECK_LAUNCH();
    return launch_cols_blue<true>(reinterpret_cast<const float2*>(spec_out), reinterpret_cast<float2*>(spec_out), nslices,
                                  H, sH, chirp, bh, st);
  }
  const size_t smem = (size_t)H * kRSmma * 8 + (size_t)2 * kC2 * kMixLd * 4 + kC2 * 4 + (size_t)H * 8;
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    constexpr int TH = (N1_ * N2_ >= 256) ? 512 : 256;                                                              \
    int rc = set_smem(fft_cols_mix_kernel<N1_, N2_, TH>, smem);                                                     \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_cols_mix_kernel<N1_, N2_, TH>, B * (W / 2 + 1), TH, smem, (cudaStream_t)stream,                  \
               reinterpret_cast<const float2*>(spec_in), reinterpret_cast<float2*>(spec_out), w, bias);             \
  }
  MTD_FFT_DISPATCH(H, CALL)
#undef CALL
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int mtd_fft_cols_mix_bwd(const float* spec_x, const float* spec_g, float* spec_out, const float* w, const float* bias,
                         float* part, float* dw, float* db, int B, int H, int W, int C, void* stream) {
  MTD_REQUIRE(spec_x && spec_g && spec_out && w && bias && part && dw && db);
  MTD_REQUIRE(B > 0 && fft_len_ok(H) && H <= 256 && fft_len_ok(W) && C == kC);   // wk below assumes an even W
  const size_t smem = (size_t)H * kRSmma * 16 + kC2 * 4 + (size_t)H * 8;
  const int Wh = W / 2 + 1, nparts = B * Wh;
  cudaStream_t st = (cudaStream_t)stream;
  float* bw = part + (size_t)nparts * (kC2 * kC2 + kC2);
  mtd_launch(fft_mix_prepare_kernel, 1, 256, 0, st, w, 1.0f / sqrtf((float)H), bw);
  MTD_CHECK_LAUNCH();
#define CALL(N1_, N2_)                                                                                              \
  {                                                                                                                 \
    int rc = set_smem(fft_cols_mix_bwd_kernel<N1_, N2_>, smem);                                                     \
    if (rc) return rc;                                                                                              \
    mtd_launch(fft_cols_mix_bwd_kernel<N1_, N2_>, nparts, kThreadsFft, smem, st, reinterpret_cast<const float2*>(spec_x), \
               reinterpret_cast<const float2*>(spec_g), reinterpret_cast<float2*>(spec_out), w, bias, part, bw, Wh, W); \
  }
  MTD_FFT_DISPATCH(H, CALL)
#undef CALL
  MTD_CHECK_LAUNCH();
  const int per = kC2 * kC2 + kC2;
  mtd_launch(fft_wgrad_reduce_kernel, (per + 31) / 32, 256, 0, st, part, nparts, dw, db);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

}  // extern "C"
