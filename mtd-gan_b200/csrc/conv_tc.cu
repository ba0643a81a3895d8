// tcgen05 / TMEM implicit-GEMM convolution for sm_100a (TF32 operands, fp32 accumulate in TMEM).
//
//   out[b,h,w,n] = epilogue( sum_t sum_c  in[b, h+dy[t], w+dx[t], c] * wp[n][t][c] )          (stride 1)
//
// GEMM view: M = B*H*W output pixels (128 per tile = one TMEM lane each), N = output channels
// (BN = 32/64/128 per tile), K = taps x channels, consumed 32 channels (128 B, one SWIZZLE_128B row) at a
// time.  No im2col buffer exists anywhere: for tap t the A tile is the TMA box
// (32 ch, TW, TH, TB) of the NHWC input at coordinates (c0, w0+dx, h0+dy, b0); the convolution halo / zero
// padding is TMA's out-of-bounds zero fill.  Two inputs (torch.cat skip connections) are two tensor maps.
//
// Persistent, warp-specialised CTA (one per SM), 10 warps:
//   warp 0      TMA producer  (one elected lane): A box + B box per k-step into a 4..6 stage smem ring
//   warp 1      MMA issuer    (one elected lane): 4 x tcgen05.mma.kind::tf32 (128 x BN x 8) per k-step,
//               tcgen05.commit frees the smem stage / publishes the accumulator; owns TMEM alloc/dealloc
//   warps 2-5   operand rounding: cvt.rna.tf32.f32 of the landed A tile in place (tcgen05 TRUNCATES fp32 to
//               tf32, a systematic bias; weights are pre-rounded by the pack kernel), fence.proxy.async
//   warps 6-9   epilogue: tcgen05.ld 32x32b of the finished accumulator (double-buffered in TMEM so it
//               overlaps the next tile's MMAs), scale(1/sigma)+bias+activation+residual adds, float4 stores
//
// Numerics, selectable per call (`passes`):
//   1  TF32 (10-bit mantissa, round-to-nearest operands), fp32 accumulation: <= 2e-3 relative.
//   3  error-compensated "3xTF32": a = a_hi + a_lo, w = w_hi + w_lo (each part TF32-exact), D += a_hi*w_hi
//      + a_lo*w_hi + a_hi*w_lo — the dropped a_lo*w_lo term is ~2^-22 relative, so the result is fp32-grade
//      (<= 1e-5 relative) at 3 MMAs per k-step.  The rounding warps produce a_lo on the fly; w_lo is
//      pre-split by mtd_split_tf32.  This is the default for training (gradient parity <= 1e-4).
// Used for forward convs and stride-1 dgrad with C % 32 == 0, N % 32 == 0 and >= 2048 output pixels;
// everything else runs on conv_simt.cu (exact fp32).
#include <cuda.h>
#include <mutex>
#include <unordered_map>
#include <string>
#include <string.h>
#include <stdlib.h>
#include "common.cuh"
#include "mtdgan_b200.h"

namespace {

constexpr int kMaxTaps = 16;
constexpr int kBM = 128;
constexpr int kABytes = kBM * 128;        // 128 rows x 32 tf32
constexpr int kThreads = 320;

struct TcArgs {
  int B, H, W, C1, C2, N;
  int T;
  int dy[kMaxTaps], dx[kMaxTaps];
  int TW, TH, TB, n_wt, n_ht, n_bt, n_nt, n_tiles;
  int kc1, kc2;                 // 32-channel chunks per source
  int stages;
  int wrows_total;              // rows of the full packed weight buffer (offset of the lo half, passes == 3)
  int ksplit, kper;             // split-K: tile = mn_tile * ksplit + ks, k-steps [ks*kper, (ks+1)*kper)
  int inH, inW, es;             // input tensor dims and conv stride (A tile = TMA box with elementStrides es)
  int m_tiles, n_groups, ra, rb; // v2 kernel: pixel tiles, groups of MT pixel tiles, raw-A / B ring depths
  int outH, outW, omy, omx, ooy, oox;   // output pixel = (h*omy+ooy, w*omx+oox) in a (B,outH,outW,N) tensor
  float* out;
  float* out2;                  // split output (dgrad of a torch.cat layer): channels [n_split, N) go to out2, n_split | BN tiles
  int n_split;                  // 0 = single output
  const float* scale;           // 1/sigma: one scalar, or (scale_group > 0) one per group of scale_group samples
  int scale_group;
  const float* bias;
  int pre_act;
  const float* add1;
  const float* add2;
  int post_act;
  const float* mask_src;
  int mask_act;
  float slope;
  float* aux;
  // v1 kernel work decomposition (see "stream-K" below): tiles [0, n_dp) are processed whole, round-robin over the
  // CTAs; the k-steps of tiles [n_dp, n_dp + sk_tiles) form one flat range cut into equal pieces of sk_per steps,
  // piece c going to CTA c, partial sums to ws[slot][128][BN] with slot = sk_tile * sk_P + (c - first CTA of the tile)
  int n_dp, sk_tiles, sk_per, sk_P;
  // stride-2 dgrad as ONE launch: n_cls = 4 output-parity classes; tile = cls * tiles_per_cls + (m, n) tile; class cls
  // uses taps dy/dx[cls*T ..], weight rows [cls*N, (cls+1)*N) of the stacked pack and output offset (cls >> 1, cls & 1)
  int n_cls, tiles_per_cls;
  float* ws;
  long long ws_floats;          // host side only: capacity of ws
  int grid;                     // host side only: CTAs to launch
};

// ---------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  int spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    if (++spins > (1 << 22)) __trap();      // a lost arrival must fail the launch, never hang the GPU
  }
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint32_t dst, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (=1, unused for swizzled K-major) | [32,46) SBO >> 4
//   (8 rows x 128 B = 1024 B) | [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6), a=b=TF32 [7,10)/[10,13), K-major both,
// N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int bn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}

__device__ __forceinline__ float tc_row_scale(const TcArgs& a, int b) {
  return a.scale ? __ldg(a.scale + (a.scale_group > 0 ? b / a.scale_group : 0)) : 1.f;
}

// scale / bias / pre-activation / aux copy / residual adds / post-activation / gradient mask of 4 consecutive
// output channels, then the store (the one epilogue of every forward / dgrad path)
__device__ __forceinline__ void tc_store4(const TcArgs& a, float* out, size_t idx, int n, float scale, float x0, float x1, float x2,
                                          float x3) {
  float o[4] = {x0 * scale, x1 * scale, x2 * scale, x3 * scale};
  if (a.bias) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(a.bias + n));
    o[0] += b.x; o[1] += b.y; o[2] += b.z; o[3] += b.w;
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = mtd_act(o[e], a.pre_act, a.slope);
  if (a.aux) *reinterpret_cast<float4*>(a.aux + idx) = make_float4(o[0], o[1], o[2], o[3]);
  if (a.add1) { float4 t = __ldg(reinterpret_cast<const float4*>(a.add1 + idx)); o[0] += t.x; o[1] += t.y; o[2] += t.z; o[3] += t.w; }
  if (a.add2) { float4 t = __ldg(reinterpret_cast<const float4*>(a.add2 + idx)); o[0] += t.x; o[1] += t.y; o[2] += t.z; o[3] += t.w; }
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = mtd_act(o[e], a.post_act, a.slope);
  if (a.mask_src) {
    float4 t = __ldg(reinterpret_cast<const float4*>(a.mask_src + idx));
    o[0] *= mtd_act_grad(t.x, a.mask_act, a.slope); o[1] *= mtd_act_grad(t.y, a.mask_act, a.slope);
    o[2] *= mtd_act_grad(t.z, a.mask_act, a.slope); o[3] *= mtd_act_grad(t.w, a.mask_act, a.slope);
  }
  *reinterpret_cast<float4*>(out + idx) = make_float4(o[0], o[1], o[2], o[3]);
}

// output tensor, row stride and first column of the tile starting at channel n0 (split outputs: see TcArgs::out2)
__device__ __forceinline__ float* tc_out_of(const TcArgs& a, int n0, int& ncols, int& nloc) {
  if (a.n_split > 0 && n0 >= a.n_split) { ncols = a.N - a.n_split; nloc = n0 - a.n_split; return a.out2; }
  ncols = a.n_split > 0 ? a.n_split : a.N; nloc = n0;
  return a.out;
}

// ---- work decomposition of the v1 kernel: data-parallel waves + one stream-K wave ---------------------------
// A layer with mn output tiles of K k-steps each runs floor(mn / #SM) full waves tile-per-CTA; the remaining
// (mn mod #SM) tiles -- or ALL tiles of a layer with fewer tiles than SMs -- are cut along K into #CTA equal pieces,
// so every SM gets the same number of k-steps (a 160-tile layer on 148 SMs takes 1.08 instead of 2 tile-times, a
// 12-tile layer gets 12-way split-K).  Pieces write raw fp32 partial tiles to the workspace with plain stores;
// tc_sk_finish_kernel adds the pieces of a tile IN ORDER (deterministic, no atomics, no memset) and runs the epilogue.
struct Work { int tile, kb, ke, slot; };
struct WorkIter {
  int dp_tile, pos, end;
  __device__ __forceinline__ WorkIter(const TcArgs& a, int K) {
    dp_tile = blockIdx.x;
    pos = (int)blockIdx.x * a.sk_per;
    end = min(pos + a.sk_per, a.sk_tiles * K);
  }
  __device__ __forceinline__ bool next(const TcArgs& a, int K, Work& w) {
    if (dp_tile < a.n_dp) {
      w.tile = dp_tile; w.kb = 0; w.ke = K; w.slot = -1;
      dp_tile += gridDim.x;
      return true;
    }
    if (pos < end) {
      const int st = pos / K;
      w.tile = a.n_dp + st;
      w.kb = pos - st * K;
      w.ke = min(K, w.kb + end - pos);
      w.slot = st * a.sk_P + ((int)blockIdx.x - (st * K) / a.sk_per);
      pos += w.ke - w.kb;
      return true;
    }
    return false;
  }
};

struct PipeState {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance(int n) {
    if (++stage == n) { stage = 0; phase ^= 1u; }
  }
};

template <int BN, int NPASS>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapA2,
               const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
               const __grid_constant__ TcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kBBytes = BN * 128;
  constexpr int kNA = NPASS == 3 ? 2 : 1;                           // A_hi (+ A_lo), B_hi (+ B_lo)
  constexpr int kStageBytes = kNA * (kABytes + kBBytes);
  constexpr int kTxBytes = kABytes + kNA * kBBytes;                 // bytes TMA writes per stage (A_lo is produced on chip)
  constexpr int kOffAlo = kABytes, kOffB = kNA * kABytes, kOffBlo = kNA * kABytes + kBBytes;
  // 3xTF32: [w_hi | w_lo] is ONE B operand of 2*BN rows, so a_hi * [w_hi | w_lo] is one N = 2*BN MMA (the A slice is read
  // from shared memory once for both products) and a_lo * w_hi a second N = BN MMA into the upper accumulator half; the
  // epilogue adds the halves.  Tensor-core operand reads per k-step: 80 KB instead of 96 KB (BN = 128).
  constexpr uint32_t kAccCols = NPASS == 3 ? 2 * BN : BN;
  constexpr uint32_t kTmemCols = (2 * kAccCols) < 32 ? 32 : 2 * kAccCols;      // two accumulators; power of two >= 32

  // 1024-byte alignment for SWIZZLE_128B
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int S = a.stages;
  const uint32_t bar_base = base + (uint32_t)S * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
  auto conv_bar = [&](int s) { return bar_base + 8u * (2 * S + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (3 * S + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (3 * S + 2 + i); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * S + 4);
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.kc1 + a.kc2;
  const int kiters = a.T * kchunks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA1);
    if (a.kc2) prefetch_tmap(&mapA2);
    prefetch_tmap(&mapB);
    if (NPASS == 3) prefetch_tmap(&mapBlo);
    for (int s = 0; s < S; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      mbar_init(conv_bar(s), 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  // barriers initialised, TMEM allocated, descriptors prefetched: all of it overlapped the previous kernel's tail
  mtd_pdl_prologue();

  auto decode_tile = [&](int tile, int& b0, int& h0, int& w0, int& n0, int& cls) {
    cls = 0;
    if (a.n_cls > 1) { cls = tile / a.tiles_per_cls; tile -= cls * a.tiles_per_cls; }
    int nt = tile % a.n_nt, m = tile / a.n_nt;
    int mw = m % a.n_wt;
    m /= a.n_wt;
    int mh = m % a.n_ht, mb = m / a.n_ht;
    b0 = mb * a.TB; h0 = mh * a.TH; w0 = mw * a.TW; n0 = nt * BN;
  };

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      PipeState st;
      WorkIter wi(a, kiters);
      Work wk;
      while (wi.next(a, kiters, wk)) {
        int b0, h0, w0, n0, cls;
        decode_tile(wk.tile, b0, h0, w0, n0, cls);
        const int nblk = (n0 >> 5) + cls * (a.N >> 5);            // weight rows of this class in the stacked pack
        for (int it = wk.kb; it < wk.ke; ++it) {
          mbar_wait(empty_bar(st.stage), st.phase ^ 1u);
          mbar_expect_tx(full_bar(st.stage), kTxBytes);
          const int t = it / kchunks, cc = it - t * kchunks, tt = cls * a.T + t;
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes, sb = sa + kOffB;
          if (cc < a.kc1) tma_load_4d(&mapA1, sa, full_bar(st.stage), cc * 32, w0 * a.es + a.dx[tt], h0 * a.es + a.dy[tt], b0);
          else tma_load_4d(&mapA2, sa, full_bar(st.stage), (cc - a.kc1) * 32, w0 * a.es + a.dx[tt], h0 * a.es + a.dy[tt], b0);
          tma_load_4d(&mapB, sb, full_bar(st.stage), 0, 0, it, nblk);             // k-step `it` == (t*Ctot + cc*32)/32
          if (NPASS == 3) tma_load_4d(&mapBlo, sa + kOffBlo, full_bar(st.stage), 0, 0, it, nblk);
          st.advance(S);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      PipeState st;
      constexpr uint32_t idesc_main = make_idesc((int)kAccCols), idesc_lo = make_idesc(BN);
      WorkIter wi(a, kiters);
      Work wk;
      for (int lt = 0; wi.next(a, kiters, wk); ++lt) {
        const int acc = lt & 1;
        const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
        const int k_begin = wk.kb, k_end = wk.ke;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * kAccCols;
        for (int it = k_begin; it < k_end; ++it) {
          mbar_wait(conv_bar(st.stage), st.phase);
          tc_fence_after();
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes;
          const uint64_t da = make_sw128_desc(sa), db = make_sw128_desc(sa + kOffB);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {      // 4 x (K = 8 tf32 = 32 B): +2 in 16-byte address units
            umma_tf32(tmem_d, da + 2u * kk, db + 2u * kk, idesc_main, (it > k_begin || kk > 0) ? 1u : 0u);
            if (NPASS == 3) {                   // cross term a_lo * w_hi into the upper half (w_lo rows follow w_hi in the stage)
              const uint64_t dal = make_sw128_desc(sa + kOffAlo);
              umma_tf32(tmem_d + BN, dal + 2u * kk, db + 2u * kk, idesc_lo, 1u);
            }
          }
          umma_commit(empty_bar(st.stage));       // implies tcgen05.fence::before_thread_sync
          st.advance(S);
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else if (warp < 6) {
    // ===== operand rounding (fp32 -> tf32, round to nearest) =====
    const int ct = threadIdx.x - 64;               // 0..127
    PipeState st;
    WorkIter wi(a, kiters);
    Work wk;
    while (wi.next(a, kiters, wk)) {
      for (int it = wk.kb; it < wk.ke; ++it) {
        mbar_wait(full_bar(st.stage), st.phase);
        uint4* tileA = reinterpret_cast<uint4*>(gen_base + (size_t)st.stage * kStageBytes);
        // Integer arithmetic instead of cvt.rna.tf32.f32 (quarter-rate: it was the k-step bound for BN <= 64):
        // (bits + 0x1000) & ~0x1fff == cvt.rna (nearest, ties away from zero).
        //   plain TF32: a_hi = rn_tf32(a) replaces the raw tile (the tensor core would TRUNCATE the raw fp32: a bias).
        //   3xTF32: the raw tile STAYS -- the tensor core's truncation IS a_hi = trunc_tf32(a) -- and only
        //   a_lo = rn_tf32(a - trunc_tf32(a)) is written (the difference is exact in fp32, so hi + lo carries no bias);
        //   one 16 KB store pass less per k-step through the shared-memory pipe that bounds this kernel.  The dropped
        //   a_lo * w_lo term is <= 2^-21 relative instead of 2^-22.
#pragma unroll 8
        for (int j = 0; j < kABytes / 16 / 128; ++j) {
          const uint4 v = tileA[ct + 128 * j];
          if (NPASS == 3) {
            uint4 l;
            l.x = (__float_as_uint(__uint_as_float(v.x) - __uint_as_float(v.x & 0xffffe000u)) + 0x1000u) & 0xffffe000u;
            l.y = (__float_as_uint(__uint_as_float(v.y) - __uint_as_float(v.y & 0xffffe000u)) + 0x1000u) & 0xffffe000u;
            l.z = (__float_as_uint(__uint_as_float(v.z) - __uint_as_float(v.z & 0xffffe000u)) + 0x1000u) & 0xffffe000u;
            l.w = (__float_as_uint(__uint_as_float(v.w) - __uint_as_float(v.w & 0xffffe000u)) + 0x1000u) & 0xffffe000u;
            tileA[kOffAlo / 16 + ct + 128 * j] = l;
          } else {
            uint4 h;
            h.x = (v.x + 0x1000u) & 0xffffe000u; h.y = (v.y + 0x1000u) & 0xffffe000u;
            h.z = (v.z + 0x1000u) & 0xffffe000u; h.w = (v.w + 0x1000u) & 0xffffe000u;
            tileA[ct + 128 * j] = h;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
        __syncwarp();
        if (lane == 0) mbar_arrive(conv_bar(st.stage));                // one arrival per rounding warp (count 4)
        st.advance(S);
      }
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;                        // TMEM lane group this warp may access
    const int r = q * 32 + lane;                   // accumulator row == pixel within the tile
    const int bl = r / (a.TH * a.TW), rem = r - bl * (a.TH * a.TW);
    const int hl = rem / a.TW, wl = rem - hl * a.TW;
    WorkIter wi(a, kiters);
    Work wk;
    for (int lt = 0; wi.next(a, kiters, wk); ++lt) {
      int b0, h0, w0, n0, cls;
      decode_tile(wk.tile, b0, h0, w0, n0, cls);
      const int ooy = a.n_cls > 1 ? (cls >> 1) : a.ooy, oox = a.n_cls > 1 ? (cls & 1) : a.oox;
      const int acc = lt & 1;
      const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int b = b0 + bl;
      const bool valid = b < a.B;
      const float scale = valid ? tc_row_scale(a, b) : 1.f;
      int ncols, nloc;
      float* outp = tc_out_of(a, n0, ncols, nloc);
      const size_t rowoff =
          (((size_t)b * a.outH + ((h0 + hl) * a.omy + ooy)) * a.outW + ((w0 + wl) * a.omx + oox)) * ncols + nloc;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * kAccCols + (uint32_t)c0;
        tmem_ld32(taddr, v);
        if (NPASS == 3) {
          uint32_t u[32];
          tmem_ld32(taddr + BN, u);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        }
        if (wk.slot >= 0) {
          // stream-K piece: raw partial sums to the workspace tile (plain stores; rows past the batch are zeros)
          float* wrow = a.ws + ((size_t)wk.slot * kBM + r) * BN + c0;
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(wrow + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                               __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        } else if (valid) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            tc_store4(a, outp, rowoff + c0 + j, n0 + c0 + j, scale, __uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                      __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}


// =====================================================================================================
// v2 forward / dgrad kernel: A operand through TENSOR MEMORY, several pixel tiles per CTA.
//
// v1 keeps A_hi / A_lo in shared memory, which (with the 3xTF32 operand doubling) leaves room for only 2-5
// pipeline stages and makes every pixel tile re-stream the weights from L2.  Here
//   * TMA lands the raw fp32 A tile (16 KB) in a deep shared-memory ring;
//   * the rounding warps read their own row (lane = pixel = TMEM lane, de-swizzled LDS.128), split it into
//     tf32 hi / lo and write it with tcgen05.st into a 2-slot A ring in TMEM — the MMA takes A from TMEM
//     (tcgen05.mma [d], [a_tmem], b_desc), so shared memory only holds raw A and the weight tiles;
//   * each weight stage (B_hi | B_lo) is used by MT pixel tiles with MT accumulators in TMEM (MT*BN columns):
//     weight traffic per FLOP drops by MT, and a skinny-M layer (<= MT pixel tiles) streams its weights once.
// TMEM budget: MT*BN accumulator columns + 2 * (32 | 64) A-ring columns <= 512.
// =====================================================================================================
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}

__device__ __forceinline__ void tc_epilogue_chunk(const TcArgs& a, const uint32_t (&v)[32], bool valid, size_t rowoff, int n0,
                                                  int c0, float scale) {
  if (valid && a.ksplit > 1) {
#pragma unroll
    for (int j = 0; j < 32; ++j) atomicAdd(a.out + rowoff + c0 + j, __uint_as_float(v[j]));
  } else if (valid) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const size_t idx = rowoff + c0 + j;
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float x = __uint_as_float(v[j + e]) * scale;
        if (a.bias) x += __ldg(a.bias + n0 + c0 + j + e);
        o[e] = mtd_act(x, a.pre_act, a.slope);
      }
      if (a.aux) *reinterpret_cast<float4*>(a.aux + idx) = make_float4(o[0], o[1], o[2], o[3]);
      if (a.add1) { float4 t = __ldg(reinterpret_cast<const float4*>(a.add1 + idx)); o[0] += t.x; o[1] += t.y; o[2] += t.z; o[3] += t.w; }
      if (a.add2) { float4 t = __ldg(reinterpret_cast<const float4*>(a.add2 + idx)); o[0] += t.x; o[1] += t.y; o[2] += t.z; o[3] += t.w; }
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = mtd_act(o[e], a.post_act, a.slope);
      if (a.mask_src) {
        float4 t = __ldg(reinterpret_cast<const float4*>(a.mask_src + idx));
        o[0] *= mtd_act_grad(t.x, a.mask_act, a.slope); o[1] *= mtd_act_grad(t.y, a.mask_act, a.slope);
        o[2] *= mtd_act_grad(t.z, a.mask_act, a.slope); o[3] *= mtd_act_grad(t.w, a.mask_act, a.slope);
      }
      *reinterpret_cast<float4*>(a.out + idx) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}

__host__ __device__ constexpr uint32_t next_pow2_cols(uint32_t c) { return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }

template <int BN, int MT, int NPASS>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapA2,
                const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
                const __grid_constant__ TcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kNB = NPASS == 3 ? 2 : 1;
  constexpr int kBBytes = kNB * BN * 128;                        // B_hi (| B_lo) per k-step
  constexpr uint32_t kACols = kNB * 32;                          // A_hi (| A_lo) columns per TMEM A slot
  constexpr uint32_t kAccCols = MT * BN;
  constexpr uint32_t kTmemCols = next_pow2_cols(kAccCols + 2 * kACols);
  static_assert(kAccCols + 2 * kACols <= 512, "TMEM budget exceeded");

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int RA = a.ra, RB = a.rb;
  const uint32_t b_base = base + (uint32_t)RA * kABytes;
  const uint32_t bar_base = b_base + (uint32_t)RB * kBBytes;
  auto rfull = [&](int s) { return bar_base + 8u * s; };
  auto rempty = [&](int s) { return bar_base + 8u * (RA + s); };
  auto bfull = [&](int s) { return bar_base + 8u * (2 * RA + s); };
  auto bempty = [&](int s) { return bar_base + 8u * (2 * RA + RB + s); };
  auto afull = [&](int s) { return bar_base + 8u * (2 * RA + 2 * RB + s); };
  auto aempty = [&](int s) { return bar_base + 8u * (2 * RA + 2 * RB + 2 + s); };
  const uint32_t tfull = bar_base + 8u * (2 * RA + 2 * RB + 4);
  const uint32_t tempty = tfull + 8u;
  const uint32_t tmem_slot = tfull + 16u;
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.kc1 + a.kc2;
  const int kiters = a.T * kchunks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA1);
    if (a.kc2) prefetch_tmap(&mapA2);
    prefetch_tmap(&mapB);
    if (NPASS == 3) prefetch_tmap(&mapBlo);
    for (int s = 0; s < RA; ++s) { mbar_init(rfull(s), 1); mbar_init(rempty(s), 4); }
    for (int s = 0; s < RB; ++s) { mbar_init(bfull(s), 1); mbar_init(bempty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(afull(s), 4); mbar_init(aempty(s), 1); }
    mbar_init(tfull, 1);
    mbar_init(tempty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  // barriers initialised, TMEM allocated, descriptors prefetched: all of it overlapped the previous kernel's tail
  mtd_pdl_prologue();
  const uint32_t tmem_a0 = tmem_base + kAccCols;

  // tile = (group * n_nt + nt) * ksplit + ks ; group g covers pixel tiles g*MT .. g*MT+MT-1
  auto decode_tile = [&](int tile, int& g, int& n0, int& k_begin, int& k_end) {
    const int ks = tile % a.ksplit;
    tile /= a.ksplit;
    k_begin = ks * a.kper;
    k_end = min(kiters, k_begin + a.kper);
    n0 = (tile % a.n_nt) * BN;
    g = tile / a.n_nt;
  };
  auto decode_mtile = [&](int mt, int& b0, int& h0, int& w0) {
    int mw = mt % a.n_wt;
    mt /= a.n_wt;
    int mh = mt % a.n_ht, mb = mt / a.n_ht;
    b0 = mb * a.TB; h0 = mh * a.TH; w0 = mw * a.TW;
  };

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      PipeState sr, sb;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int g, n0, k_begin, k_end;
        decode_tile(tile, g, n0, k_begin, k_end);
        for (int it = k_begin; it < k_end; ++it) {
          const int t = it / kchunks, cc = it - t * kchunks;
          mbar_wait(bempty(sb.stage), sb.phase ^ 1u);
          mbar_expect_tx(bfull(sb.stage), kBBytes);
          const uint32_t sbm = b_base + (uint32_t)sb.stage * kBBytes;
          tma_load_4d(&mapB, sbm, bfull(sb.stage), 0, 0, it, n0 >> 5);               // k-step `it` == (t*Ctot + cc*32)/32
          if (NPASS == 3) tma_load_4d(&mapBlo, sbm + BN * 128, bfull(sb.stage), 0, 0, it, n0 >> 5);
          sb.advance(RB);
#pragma unroll 1
          for (int j = 0; j < MT; ++j) {
            const int mt = g * MT + j;
            if (mt >= a.m_tiles) break;
            int b0, h0, w0;
            decode_mtile(mt, b0, h0, w0);
            mbar_wait(rempty(sr.stage), sr.phase ^ 1u);
            mbar_expect_tx(rfull(sr.stage), kABytes);
            const uint32_t sam = base + (uint32_t)sr.stage * kABytes;
            if (cc < a.kc1) tma_load_4d(&mapA1, sam, rfull(sr.stage), cc * 32, w0 * a.es + a.dx[t], h0 * a.es + a.dy[t], b0);
            else tma_load_4d(&mapA2, sam, rfull(sr.stage), (cc - a.kc1) * 32, w0 * a.es + a.dx[t], h0 * a.es + a.dy[t], b0);
            sr.advance(RA);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: A from TMEM, B from shared memory =====
    if (lane == 0) {
      PipeState sb, sa;
      constexpr uint32_t idesc = make_idesc(BN);
      int lt = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
        int g, n0, k_begin, k_end;
        decode_tile(tile, g, n0, k_begin, k_end);
        mbar_wait(tempty, ((uint32_t)lt & 1u) ^ 1u);
        tc_fence_after();
        for (int it = k_begin; it < k_end; ++it) {
          mbar_wait(bfull(sb.stage), sb.phase);
          const uint32_t sbm = b_base + (uint32_t)sb.stage * kBBytes;
          const uint64_t db = make_sw128_desc(sbm), dbl = make_sw128_desc(sbm + BN * 128);
#pragma unroll 1
          for (int j = 0; j < MT; ++j) {
            if (g * MT + j >= a.m_tiles) break;
            mbar_wait(afull(sa.stage), sa.phase);
            tc_fence_after();
            const uint32_t a_hi = tmem_a0 + (uint32_t)sa.stage * kACols, a_lo = a_hi + 32;
            const uint32_t d = tmem_base + (uint32_t)(j * BN);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              const uint32_t accum = (it > k_begin || kk > 0) ? 1u : 0u;
              if (NPASS == 3) {
                umma_tf32_ts(d, a_lo + 8u * kk, db + 2u * kk, idesc, accum);
                umma_tf32_ts(d, a_hi + 8u * kk, dbl + 2u * kk, idesc, 1u);
                umma_tf32_ts(d, a_hi + 8u * kk, db + 2u * kk, idesc, 1u);
              } else {
                umma_tf32_ts(d, a_hi + 8u * kk, db + 2u * kk, idesc, accum);
              }
            }
            umma_commit(aempty(sa.stage));
            sa.advance(2);
          }
          umma_commit(bempty(sb.stage));
          sb.advance(RB);
        }
        umma_commit(tfull);
      }
    }
  } else if (warp < 6) {
    // ===== operand split: own row of the raw A tile -> tf32 hi / lo -> TMEM =====
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    PipeState sr, sa;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      int g, n0, k_begin, k_end;
      decode_tile(tile, g, n0, k_begin, k_end);
      for (int it = k_begin; it < k_end; ++it) {
#pragma unroll 1
        for (int j = 0; j < MT; ++j) {
          if (g * MT + j >= a.m_tiles) break;
          mbar_wait(rfull(sr.stage), sr.phase);
          const unsigned char* rowp = gen_base + (size_t)sr.stage * kABytes + (size_t)row * 128;
          uint32_t hi[32], lo[32];
#pragma unroll
          for (int c = 0; c < 8; ++c) {                 // logical 16-byte chunk c lives at physical chunk c ^ (row & 7)
            const float4 v = *reinterpret_cast<const float4*>(rowp + ((c ^ (row & 7)) << 4));
            const float f[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              uint32_t h;
              asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(f[e]));
              hi[c * 4 + e] = h;
              if (NPASS == 3) {
                uint32_t l;
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(f[e] - __uint_as_float(h)));
                lo[c * 4 + e] = l;
              }
            }
          }
          mbar_wait(aempty(sa.stage), sa.phase ^ 1u);     // the MMAs that read this TMEM slot have completed
          tc_fence_after();
          const uint32_t ta = tmem_a0 + lane_addr + (uint32_t)sa.stage * kACols;
          tmem_st32(ta, hi);
          if (NPASS == 3) tmem_st32(ta + 32, lo);
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(rempty(sr.stage));                // raw slot may be refilled by TMA
            mbar_arrive(afull(sa.stage));
          }
          sr.advance(RA);
          sa.advance(2);
        }
      }
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int bl = r / (a.TH * a.TW), rem = r - bl * (a.TH * a.TW);
    const int hl = rem / a.TW, wl = rem - hl * a.TW;
    int lt = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
      int g, n0, k_begin, k_end;
      decode_tile(tile, g, n0, k_begin, k_end);
      mbar_wait(tfull, (uint32_t)lt & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int j = 0; j < MT; ++j) {
        const int mt = g * MT + j;
        if (mt >= a.m_tiles) break;
        int b0, h0, w0;
        decode_mtile(mt, b0, h0, w0);
        const int b = b0 + bl;
        const bool valid = b < a.B;
        const float scale = valid ? tc_row_scale(a, b) : 1.f;
        const size_t rowoff =
            (((size_t)b * a.outH + ((h0 + hl) * a.omy + a.ooy)) * a.outW + ((w0 + wl) * a.omx + a.oox)) * a.N + n0;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * BN + c0), v);
          tc_epilogue_chunk(a, v, valid, rowoff, n0, c0, scale);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// second phase of a split-K launch: `out` holds raw sums over a dense (B,outH,outW,N) tensor
__global__ void tc_finish_kernel(const __grid_constant__ TcArgs a, size_t total) {
  mtd_pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  const size_t per_sample = (size_t)a.outH * a.outW * a.N;
  for (; i < total; i += stride) {
    int n = (int)(i % a.N);
    float x = a.out[i] * tc_row_scale(a, (int)(i / per_sample));
    if (a.bias) x += __ldg(a.bias + n);
    x = mtd_act(x, a.pre_act, a.slope);
    if (a.aux) a.aux[i] = x;
    if (a.add1) x += __ldg(a.add1 + i);
    if (a.add2) x += __ldg(a.add2 + i);
    x = mtd_act(x, a.post_act, a.slope);
    if (a.mask_src) x *= mtd_act_grad(__ldg(a.mask_src + i), a.mask_act, a.slope);
    a.out[i] = x;
  }
}

// =====================================================================================================
// 32 -> 32 channel 3x3 layers (every spatial conv of the Res-FFT-Conv generator: 22 encoder / decoder layers and 21
// `img_conv`s, forward and data gradient; ALL of inference): halo-tile kernel.
//
// The general kernel above streams, per 128-pixel tile, nine tap-shifted 16 KB A boxes plus nine hi|lo weight tiles
// from L2 (216 KB) and rounds each box in shared memory.  Here
//   * the 72 KB hi|lo weight of the layer is loaded ONCE per CTA and stays resident in shared memory;
//   * one TMA box lands the (16+2) x (8+2) pixel HALO of a 16 x 8 pixel tile (23 KB, raw fp32, SWIZZLE_128B);
//   * four conversion warps split it ONCE into tf32 hi / lo planes laid out [8 chunks of 4 channels][180 halo pixels]
//     [16 B] -- the no-swizzle K-major ("interleaved") UMMA layout: a core matrix is 8 consecutive halo pixels x 16 B,
//     LBO = plane stride (2880 B), SBO = one halo row (10 pixels = 160 B);
//   * the nine taps are nine DESCRIPTOR START ADDRESSES into the same planes (shift by (dy*10 + dx) * 16 B): no data
//     moves for a tap;
//   * B_hi | B_lo of a tap are adjacent 4 KB tiles, i.e. one N = 64 operand: one MMA gives a_hi*w_hi (columns 0-31) and
//     a_hi*w_lo (columns 32-63), a second N = 32 MMA adds a_lo*w_hi to columns 32-63; the epilogue sums the halves
//     (small terms are accumulated separately from the main product).
// L2 -> SM traffic per tile: 23 KB instead of 216 KB; conversion work 1440 instead of 9216 float4 per tile.
// =====================================================================================================
constexpr int kHaloW = 10, kHaloH = 18, kHaloPix = kHaloW * kHaloH;            // halo of a 16 x 8 tile
constexpr int kRawBytes = kHaloPix * 128;                                      // 23040
constexpr int kRawStage = (kRawBytes + 1023) & ~1023;                          // 23552 (SWIZZLE_128B: 1024-aligned stages)
constexpr int kPlaneBytes = kHaloPix * 16;                                     // 2880: one 4-channel chunk of all halo pixels
constexpr int kCvStage = 2 * 8 * kPlaneBytes;                                  // hi planes | lo planes = 46080
constexpr int kC32WBytes = 9 * 2 * 4096;                                       // 9 taps x (hi | lo) 32 x 32 tiles

// no-swizzle K-major descriptor: [0,14) start >> 4 | [16,30) LBO >> 4 (between the two 16-byte K chunks of one MMA)
// | [32,46) SBO >> 4 (between 8-row groups) | version 1 | layout 0
__device__ __forceinline__ uint64_t make_interleave_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46);
}

template <int NPASS>
__global__ void __launch_bounds__(kThreads, 1)
conv_c32_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const __grid_constant__ CUtensorMap mapBlo, const __grid_constant__ TcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kNA = NPASS == 3 ? 2 : 1;
  constexpr uint32_t kAccCols = NPASS == 3 ? 64 : 32;
  constexpr uint32_t kTmemCols = 2 * kAccCols;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = base;                                      // [tap][hi 4 KB | lo 4 KB]
  const uint32_t raw_base = w_base + kC32WBytes;                     // 2 raw halo stages
  const uint32_t cv_base = raw_base + 2 * kRawStage;                 // 2 converted stages (hi planes | lo planes)
  const uint32_t bar_base = cv_base + 2 * kCvStage;
  const uint32_t wfull = bar_base;
  auto rfull = [&](int s) { return bar_base + 8u * (1 + s); };
  auto rempty = [&](int s) { return bar_base + 8u * (3 + s); };
  auto cfull = [&](int s) { return bar_base + 8u * (5 + s); };
  auto cempty = [&](int s) { return bar_base + 8u * (7 + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (9 + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (11 + i); };
  const uint32_t tmem_slot = bar_base + 8u * 13;
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA);
    prefetch_tmap(&mapB);
    if (NPASS == 3) prefetch_tmap(&mapBlo);
    mbar_init(wfull, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(rfull(s), 1);
      mbar_init(rempty(s), 4);
      mbar_init(cfull(s), 4);
      mbar_init(cempty(s), 1);
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  mtd_pdl_prologue();

  const int tiles_per_img = a.n_ht * a.n_wt;
  auto decode = [&](int tile, int& b, int& h0, int& w0) {
    b = tile / tiles_per_img;
    const int r = tile - b * tiles_per_img;
    const int th = r / a.n_wt;
    h0 = th * 16; w0 = (r - th * a.n_wt) * 8;
  };

  if (warp == 0) {
    // ===== TMA producer: the weights once, then one halo box per tile =====
    if (lane == 0) {
      mbar_expect_tx(wfull, kNA * 9 * 4096);
      for (int t = 0; t < 9; ++t) {
        tma_load_4d(&mapB, w_base + (uint32_t)t * 8192u, wfull, 0, 0, t, 0);
        if (NPASS == 3) tma_load_4d(&mapBlo, w_base + (uint32_t)t * 8192u + 4096u, wfull, 0, 0, t, 0);
      }
      PipeState st;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int b, h0, w0;
        decode(tile, b, h0, w0);
        mbar_wait(rempty(st.stage), st.phase ^ 1u);
        mbar_expect_tx(rfull(st.stage), kRawBytes);
        tma_load_4d(&mapA, raw_base + (uint32_t)st.stage * kRawStage, rfull(st.stage), 0, w0 - 1, h0 - 1, b);
        st.advance(2);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      PipeState st;
      constexpr uint32_t idesc_main = make_idesc(NPASS == 3 ? 64 : 32), idesc_lo = make_idesc(32);
      // All descriptors are precomputed: the issuing thread is ONE lane, every integer instruction in its loop costs a
      // full dependent-issue latency.  Per tap: the B descriptor and the halo shift (in 16-byte descriptor units).
      uint32_t shift16[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) shift16[t] = (uint32_t)((a.dy[t] + 1) * kHaloW + (a.dx[t] + 1));
      const uint64_t db0 = make_sw128_desc(w_base);
      const uint64_t da_stage[2] = {make_interleave_desc(cv_base, kPlaneBytes, kHaloW * 16),
                                    make_interleave_desc(cv_base + kCvStage, kPlaneBytes, kHaloW * 16)};
      mbar_wait(wfull, 0);
      int lt = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
        const int acc = lt & 1;
        const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        mbar_wait(cfull(st.stage), st.phase);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * kAccCols;
        const uint64_t da_hi = st.stage ? da_stage[1] : da_stage[0];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          // start-address field arithmetic (16-byte units): + tap shift, + 2 planes per K = 8 slice; the lo planes
          // follow the 8 hi planes; the B tile of tap t is 8 KB further, its K slices 32 B apart
          const uint64_t dat = da_hi + shift16[t];
          const uint64_t dbt = db0 + (uint64_t)(t * (8192 >> 4));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            umma_tf32(tmem_d, dat + (uint64_t)(kk * (2 * kPlaneBytes >> 4)), dbt + 2u * kk, idesc_main, (t > 0 || kk > 0) ? 1u : 0u);
            if (NPASS == 3)
              umma_tf32(tmem_d + 32u, dat + (uint64_t)((8 + 2 * kk) * (kPlaneBytes >> 4)), dbt + 2u * kk, idesc_lo, 1u);
          }
        }
        umma_commit(cempty(st.stage));
        umma_commit(tfull_bar(acc));
        st.advance(2);
      }
    }
  } else if (warp < 6) {
    // ===== operand split: raw halo (pixel-major, swizzled) -> tf32 hi / lo planes (chunk-major) =====
    const int ct = threadIdx.x - 64;               // 0..127
    PipeState sr, sc;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      mbar_wait(rfull(sr.stage), sr.phase);
      mbar_wait(cempty(sc.stage), sc.phase ^ 1u);
      const unsigned char* raw = gen_base + (raw_base - base) + (size_t)sr.stage * kRawStage;
      unsigned char* hip = gen_base + (cv_base - base) + (size_t)sc.stage * kCvStage;
      unsigned char* lop = hip + 8 * kPlaneBytes;
#pragma unroll 4
      for (int i = ct; i < 8 * kHaloPix; i += 128) {
        const int kc = i / kHaloPix, p = i - kc * kHaloPix;           // consecutive lanes: consecutive halo pixels, same chunk
        const uint4 v = *reinterpret_cast<const uint4*>(raw + (size_t)p * 128 + ((kc ^ (p & 7)) << 4));
        uint4 h;
        h.x = (v.x + 0x1000u) & 0xffffe000u; h.y = (v.y + 0x1000u) & 0xffffe000u;
        h.z = (v.z + 0x1000u) & 0xffffe000u; h.w = (v.w + 0x1000u) & 0xffffe000u;
        *reinterpret_cast<uint4*>(hip + (size_t)kc * kPlaneBytes + (size_t)p * 16) = h;
        if (NPASS == 3) {
          uint4 l;
          l.x = (__float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) + 0x1000u) & 0xffffe000u;
          l.y = (__float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) + 0x1000u) & 0xffffe000u;
          l.z = (__float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) + 0x1000u) & 0xffffe000u;
          l.w = (__float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) + 0x1000u) & 0xffffe000u;
          *reinterpret_cast<uint4*>(lop + (size_t)kc * kPlaneBytes + (size_t)p * 16) = l;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(cfull(sc.stage));
        mbar_arrive(rempty(sr.stage));
      }
      sr.advance(2);
      sc.advance(2);
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;
    const int r = q * 32 + lane;                   // accumulator row: pixel (hl, wl) = (r / 8, r % 8) of the tile
    const int hl = r >> 3, wl = r & 7;
    int lt = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
      int b, h0, w0;
      decode(tile, b, h0, w0);
      const int acc = lt & 1;
      const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
      // residual operands of this lane's output row are fetched BEFORE the accumulator is waited for: eight dependent
      // global round trips per tile would otherwise sit on the epilogue's critical path
      const float scale = tc_row_scale(a, b);
      const size_t rowoff = (((size_t)b * a.H + (h0 + hl)) * a.W + (w0 + wl)) * 32;
      float4 r1[8], r2[8];
      const bool has1 = a.add1 != nullptr, has2 = a.add2 != nullptr;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        r1[j] = has1 ? __ldg(reinterpret_cast<const float4*>(a.add1 + rowoff) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        r2[j] = has2 ? __ldg(reinterpret_cast<const float4*>(a.add2 + rowoff) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * kAccCols, v);
      if (NPASS == 3) {
        uint32_t u[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * kAccCols + 32u, u);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));            // accumulator is in registers: the next tile may overwrite it
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float o[4] = {__uint_as_float(v[4 * j]) * scale, __uint_as_float(v[4 * j + 1]) * scale, __uint_as_float(v[4 * j + 2]) * scale,
                      __uint_as_float(v[4 * j + 3]) * scale};
        if (a.bias) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(a.bias) + j);
          o[0] += bb.x; o[1] += bb.y; o[2] += bb.z; o[3] += bb.w;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = mtd_act(o[e], a.pre_act, a.slope);
        if (a.aux) *(reinterpret_cast<float4*>(a.aux + rowoff) + j) = make_float4(o[0], o[1], o[2], o[3]);
        o[0] += r1[j].x + r2[j].x; o[1] += r1[j].y + r2[j].y; o[2] += r1[j].z + r2[j].z; o[3] += r1[j].w + r2[j].w;
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = mtd_act(o[e], a.post_act, a.slope);
        if (a.mask_src) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(a.mask_src + rowoff) + j);
          o[0] *= mtd_act_grad(t.x, a.mask_act, a.slope); o[1] *= mtd_act_grad(t.y, a.mask_act, a.slope);
          o[2] *= mtd_act_grad(t.z, a.mask_act, a.slope); o[3] *= mtd_act_grad(t.w, a.mask_act, a.slope);
        }
        *(reinterpret_cast<float4*>(a.out + rowoff) + j) = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// =====================================================================================================
// General 3x3 / stride-1 layers (any multiple of 32 input channels from one or two sources, Cout tile BN = 32/64/128):
// the halo-tile scheme of conv_c32_kernel with the weights STREAMED instead of resident -- every 3x3 layer of the
// U-Net discriminator at 16x16 ... 64x64 resolution, forward and data gradient.
//
// The tap-streaming kernel (conv_tc_kernel) is bound by shared-memory bandwidth (ncu: tensor-core operand reads 46 % +
// LSU 40 % of the data pipe, tensor pipe 48 % busy): per 32-channel k-step it moves 192 KB through shared memory -- 48 KB
// of TMA writes, 48 KB of operand splitting (the SAME pixels re-split for each of the nine taps) and 96 KB of tensor-core
// reads.  Here, per 32-channel chunk of a 16 x 8 pixel tile,
//   * ONE halo box (18 x 10 pixels, 23 KB) is loaded and split ONCE into tf32 hi / lo planes; its nine taps are nine
//     descriptor start addresses (see conv_c32_kernel): operand-split traffic and A loads drop 9 x 128 / 180 = 6.4-fold;
//   * the hi | lo weight tile of a (chunk, tap) is ONE B operand of 2*BN rows: a_hi * [w_hi | w_lo] is one N = 2*BN MMA
//     (the A slice is read once for both products), a_lo * w_hi a second N = BN MMA into the upper accumulator half;
//     the epilogue adds the halves.  Tensor-core operand reads per k-step: 80 KB instead of 96 KB (BN = 128).
// Shared-memory traffic per k-step: ~120 KB instead of 192 KB; L2 -> SM traffic 34.6 KB instead of 48 KB.
// k index of this kernel: it = chunk * 9 + tap (chunk-major: a halo is used for nine consecutive k-steps); the work
// decomposition (whole tiles + one stream-K wave, tc_sk_finish_kernel) is the one of conv_tc_kernel.
// =====================================================================================================
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}

// chunk segments of a CTA's work list, in order: (tile, chunk = it / 9, taps [it % 9, ...)) -- one halo each
struct SegIter {
  WorkIter wi;
  Work wk;
  int it;
  bool ok;
  __device__ __forceinline__ SegIter(const TcArgs& a, int K) : wi(a, K) {
    ok = wi.next(a, K, wk);
    it = ok ? wk.kb : 0;
  }
  __device__ __forceinline__ void advance(const TcArgs& a, int K) {
    it = (it / 9 + 1) * 9;
    if (it >= wk.ke) {
      ok = wi.next(a, K, wk);
      it = ok ? wk.kb : 0;
    }
  }
};

template <int BN, int NPASS>
__global__ void __launch_bounds__(kThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapA2,
                 const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
                 const __grid_constant__ TcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kNA = NPASS == 3 ? 2 : 1;
  constexpr int kBStage = kNA * BN * 128;                            // [w_hi | w_lo] of one (chunk, tap)
  constexpr uint32_t kAccCols = NPASS == 3 ? 2 * BN : BN;            // main | cross-term accumulator
  constexpr uint32_t kTmemCols = 2 * kAccCols < 32 ? 32 : 2 * kAccCols;
  const int R = a.ra, S = a.stages;                                  // raw halo stages (1 or 2), weight ring depth
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t raw_base = base;
  const uint32_t cv_base = raw_base + (uint32_t)R * kRawStage;       // 2 split stages (8 hi planes | 8 lo planes)
  const uint32_t b_base = cv_base + 2u * kCvStage;                   // kCvStage = 45 * 1024: 1024-aligned
  const uint32_t bar_base = b_base + (uint32_t)S * kBStage;
  auto rfull = [&](int s) { return bar_base + 8u * s; };
  auto rempty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto cfull = [&](int s) { return bar_base + 8u * (4 + s); };
  auto cempty = [&](int s) { return bar_base + 8u * (6 + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (8 + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (10 + i); };
  auto bfull = [&](int s) { return bar_base + 8u * (12 + s); };
  auto bempty = [&](int s) { return bar_base + 8u * (12 + S + s); };
  const uint32_t tmem_slot = bar_base + 8u * (12 + 2 * S);
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.kc1 + a.kc2;
  const int kiters = 9 * kchunks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA1);
    if (a.kc2) prefetch_tmap(&mapA2);
    prefetch_tmap(&mapB);
    if (NPASS == 3) prefetch_tmap(&mapBlo);
    for (int s = 0; s < 2; ++s) {
      mbar_init(rfull(s), 1);
      mbar_init(rempty(s), 4);
      mbar_init(cfull(s), 4);
      mbar_init(cempty(s), 1);
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 4);
    }
    for (int s = 0; s < S; ++s) {
      mbar_init(bfull(s), 1);
      mbar_init(bempty(s), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  mtd_pdl_prologue();

  // tile -> (sample, first row, first column, first output channel); pixel tiles are 16 rows x 8 columns of one sample
  auto decode_tile = [&](int tile, int& b, int& h0, int& w0, int& n0) {
    const int nt = tile % a.n_nt;
    int m = tile / a.n_nt;
    const int mw = m % a.n_wt;
    m /= a.n_wt;
    const int mh = m % a.n_ht;
    b = m / a.n_ht; h0 = mh * 16; w0 = mw * 8; n0 = nt * BN;
  };

  if (warp == 0) {
    // ===== TMA producer: weight tiles in k order; halo boxes as early as the raw stages allow =====
    if (lane == 0) {
      SegIter hs(a, kiters);
      PipeState hr, bs;
      int issued = 0, needed = 0;
      auto issue_halo = [&]() {             // caller has made sure (or accepts waiting until) the raw stage is free
        int b, h0, w0, n0;
        decode_tile(hs.wk.tile, b, h0, w0, n0);
        const int cc = hs.it / 9;
        mbar_wait(rempty(hr.stage), hr.phase ^ 1u);
        mbar_expect_tx(rfull(hr.stage), kRawBytes);
        const uint32_t dst = raw_base + (uint32_t)hr.stage * kRawStage;
        if (cc < a.kc1) tma_load_4d(&mapA1, dst, rfull(hr.stage), cc * 32, w0 - 1, h0 - 1, b);
        else tma_load_4d(&mapA2, dst, rfull(hr.stage), (cc - a.kc1) * 32, w0 - 1, h0 - 1, b);
        hr.advance(R);
        hs.advance(a, kiters);
        ++issued;
      };
      WorkIter wi(a, kiters);
      Work wk;
      while (wi.next(a, kiters, wk)) {
        int b, h0, w0, n0;
        decode_tile(wk.tile, b, h0, w0, n0);
        const int nblk = n0 >> 5;
        for (int it = wk.kb; it < wk.ke; ++it) {
          const int cc = it / 9, t = it - cc * 9;
          if (it == wk.kb || t == 0) {
            ++needed;                                              // the MMA cannot pass this k-step without its halo
            while (issued < needed) issue_halo();
          } else if (hs.ok && mbar_test(rempty(hr.stage), hr.phase ^ 1u)) {
            issue_halo();                                          // a raw stage is free: prefetch the next chunk's halo
          }
          mbar_wait(bempty(bs.stage), bs.phase ^ 1u);
          mbar_expect_tx(bfull(bs.stage), kBStage);
          const uint32_t sb = b_base + (uint32_t)bs.stage * kBStage;
          tma_load_4d(&mapB, sb, bfull(bs.stage), 0, 0, t * kchunks + cc, nblk);
          if (NPASS == 3) tma_load_4d(&mapBlo, sb + BN * 128, bfull(bs.stage), 0, 0, t * kchunks + cc, nblk);
          bs.advance(S);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      PipeState cs, bs;
      constexpr uint32_t idesc_main = make_idesc((int)kAccCols), idesc_lo = make_idesc(BN);
      const uint64_t da_stage[2] = {make_interleave_desc(cv_base, kPlaneBytes, kHaloW * 16),
                                    make_interleave_desc(cv_base + kCvStage, kPlaneBytes, kHaloW * 16)};
      uint64_t da_hi = da_stage[0];
      WorkIter wi(a, kiters);
      Work wk;
      for (int lt = 0; wi.next(a, kiters, wk); ++lt) {
        const int acc = lt & 1;
        const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * kAccCols;
        for (int it = wk.kb; it < wk.ke; ++it) {
          const int cc = it / 9, t = it - cc * 9;
          if (it == wk.kb || t == 0) {
            mbar_wait(cfull(cs.stage), cs.phase);
            da_hi = cs.stage ? da_stage[1] : da_stage[0];
          }
          mbar_wait(bfull(bs.stage), bs.phase);
          tc_fence_after();
          // descriptor start-address arithmetic in 16-byte units: + tap shift, + 2 planes per K = 8 slice, lo planes after
          // the 8 hi planes; the K slices of the weight tile are 32 B apart
          const uint64_t dat = da_hi + (uint64_t)((a.dy[t] + 1) * kHaloW + (a.dx[t] + 1));
          const uint64_t dbt = make_sw128_desc(b_base + (uint32_t)bs.stage * kBStage);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            umma_tf32(tmem_d, dat + (uint64_t)(kk * (2 * kPlaneBytes >> 4)), dbt + 2u * kk, idesc_main, (it > wk.kb || kk > 0) ? 1u : 0u);
            if (NPASS == 3)
              umma_tf32(tmem_d + BN, dat + (uint64_t)((8 + 2 * kk) * (kPlaneBytes >> 4)), dbt + 2u * kk, idesc_lo, 1u);
          }
          umma_commit(bempty(bs.stage));
          bs.advance(S);
          if (it == wk.ke - 1 || t == 8) {
            umma_commit(cempty(cs.stage));
            cs.advance(2);
          }
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else if (warp < 6) {
    // ===== operand split: raw halo (pixel-major, swizzled) -> tf32 hi / lo planes (chunk-major), once per chunk segment =====
    const int ct = threadIdx.x - 64;               // 0..127
    PipeState sr, sc;
    for (SegIter sg(a, kiters); sg.ok; sg.advance(a, kiters)) {
      mbar_wait(rfull(sr.stage), sr.phase);
      mbar_wait(cempty(sc.stage), sc.phase ^ 1u);
      const unsigned char* raw = gen_base + (raw_base - base) + (size_t)sr.stage * kRawStage;
      unsigned char* hip = gen_base + (cv_base - base) + (size_t)sc.stage * kCvStage;
      unsigned char* lop = hip + 8 * kPlaneBytes;
#pragma unroll 4
      for (int i = ct; i < 8 * kHaloPix; i += 128) {
        const int kc = i / kHaloPix, p = i - kc * kHaloPix;           // consecutive lanes: consecutive halo pixels, same chunk
        const uint4 v = *reinterpret_cast<const uint4*>(raw + (size_t)p * 128 + ((kc ^ (p & 7)) << 4));
        uint4 h;
        h.x = (v.x + 0x1000u) & 0xffffe000u; h.y = (v.y + 0x1000u) & 0xffffe000u;
        h.z = (v.z + 0x1000u) & 0xffffe000u; h.w = (v.w + 0x1000u) & 0xffffe000u;
        *reinterpret_cast<uint4*>(hip + (size_t)kc * kPlaneBytes + (size_t)p * 16) = h;
        if (NPASS == 3) {
          uint4 l;
          l.x = (__float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) + 0x1000u) & 0xffffe000u;
          l.y = (__float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) + 0x1000u) & 0xffffe000u;
          l.z = (__float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) + 0x1000u) & 0xffffe000u;
          l.w = (__float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) + 0x1000u) & 0xffffe000u;
          *reinterpret_cast<uint4*>(lop + (size_t)kc * kPlaneBytes + (size_t)p * 16) = l;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(cfull(sc.stage));
        mbar_arrive(rempty(sr.stage));
      }
      sr.advance(R);
      sc.advance(2);
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;                        // TMEM lane group this warp may access
    const int r = q * 32 + lane;                   // accumulator row: pixel (hl, wl) = (r / 8, r % 8) of the tile
    const int hl = r >> 3, wl = r & 7;
    WorkIter wi(a, kiters);
    Work wk;
    for (int lt = 0; wi.next(a, kiters, wk); ++lt) {
      int b, h0, w0, n0;
      decode_tile(wk.tile, b, h0, w0, n0);
      const int acc = lt & 1;
      const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const float scale = tc_row_scale(a, b);
      int ncols, nloc;
      float* outp = tc_out_of(a, n0, ncols, nloc);
      const size_t rowoff = (((size_t)b * a.outH + (h0 + hl)) * a.outW + (w0 + wl)) * ncols + nloc;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * kAccCols + (uint32_t)c0;
        tmem_ld32(taddr, v);
        if (NPASS == 3) {
          uint32_t u[32];
          tmem_ld32(taddr + BN, u);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        }
        if (wk.slot >= 0) {
          float* wrow = a.ws + ((size_t)wk.slot * kBM + r) * BN + c0;
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(wrow + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                               __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            tc_store4(a, outp, rowoff + c0 + j, n0 + c0 + j, scale, __uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                      __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// second phase of a stream-K launch (v1 kernel): out tile = epilogue( sum over the tile's pieces, in piece order ).
// One thread per 4 output channels of one tile row; consecutive threads walk a row, so workspace reads and output
// writes are coalesced.
__global__ void __launch_bounds__(256) tc_sk_finish_kernel(const __grid_constant__ TcArgs a, int BN, int K) {
  mtd_pdl_prologue();
  const int c4n = BN >> 2;
  const long long total = (long long)a.sk_tiles * kBM * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) * 4;
    const int r = (int)((i / c4n) % kBM);
    const int st = (int)(i / ((long long)c4n * kBM));
    const int first = (st * K) / a.sk_per, last = ((st + 1) * K - 1) / a.sk_per;
    int tile = a.n_dp + st, cls = 0;
    if (a.n_cls > 1) { cls = tile / a.tiles_per_cls; tile -= cls * a.tiles_per_cls; }
    const int ooy = a.n_cls > 1 ? (cls >> 1) : a.ooy, oox = a.n_cls > 1 ? (cls & 1) : a.oox;
    const int nt = tile % a.n_nt;
    int m = tile / a.n_nt;
    const int mw = m % a.n_wt;
    m /= a.n_wt;
    const int mh = m % a.n_ht, mb = m / a.n_ht;
    const int bl = r / (a.TH * a.TW), rem = r - bl * (a.TH * a.TW);
    const int hl = rem / a.TW, wl = rem - hl * a.TW;
    const int b = mb * a.TB + bl;
    if (b >= a.B) continue;
    const float* wsp = a.ws + ((size_t)st * a.sk_P * kBM + r) * BN + c;
    float4 sum = __ldcg(reinterpret_cast<const float4*>(wsp));
    // four pieces in flight per thread (a dependent add after every load made the pass a chain of L2 latencies); the
    // pieces are still ADDED strictly in order
    const int P = last - first + 1;
    for (int p = 1; p < P; p += 4) {
      float4 t[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        t[q] = p + q < P ? __ldcg(reinterpret_cast<const float4*>(wsp + (size_t)(p + q) * kBM * BN)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (p + q < P) { sum.x += t[q].x; sum.y += t[q].y; sum.z += t[q].z; sum.w += t[q].w; }
    }
    int ncols, nloc;
    float* outp = tc_out_of(a, nt * BN, ncols, nloc);
    const size_t rowoff = (((size_t)b * a.outH + ((mh * a.TH + hl) * a.omy + ooy)) * a.outW +
                           ((mw * a.TW + wl) * a.omx + oox)) * ncols + nloc;
    tc_store4(a, outp, rowoff + c, nt * BN + c, tc_row_scale(a, b), sum.x, sum.y, sum.z, sum.w);
  }
}

// ---------------------------------------------------------------------------------------------------
// host side: tensor maps
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

std::mutex g_map_mutex;
std::unordered_map<std::string, CUtensorMap> g_map_cache;

// activations: rank-4 (C, W, H, B) fp32, box (32, TW, TH, TB), OOB -> zeros.  atom32 = false: SWIZZLE_128B
// (K-major operands of the forward / dgrad kernels); atom32 = true: SWIZZLE_128B_ATOM_32B (MN-major tf32
// operands of the wgrad kernel)
// es = conv stride: the box traverses es*TW x es*TH input pixels with elementStrides (1, es, es, 1), i.e. it lands
// exactly the TW x TH pixels a strided convolution tap needs.
int make_act_map(CUtensorMap* out, const float* ptr, int C, int W, int H, int B, int TW, int TH, int TB, bool atom32 = false,
                 int es = 1) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return MTD_EINVAL;
  char keybuf[128];
  snprintf(keybuf, sizeof(keybuf), "A%d%d%p:%d:%d:%d:%d:%d:%d:%d", (int)atom32, es, (const void*)ptr, C, W, H, B, TW, TH, TB);
  std::string key(keybuf);
  {
    std::lock_guard<std::mutex> lk(g_map_mutex);
    auto it = g_map_cache.find(key);
    if (it != g_map_cache.end()) { *out = it->second; return MTD_OK; }
  }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)(TW * es), (cuuint32_t)(TH * es), (cuuint32_t)TB};
  cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
  if (box[1] > 256 || box[2] > 256) return MTD_EINVAL;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return MTD_EINVAL;
  std::lock_guard<std::mutex> lk(g_map_mutex);
  if (g_map_cache.size() > 8192) g_map_cache.clear();
  g_map_cache[key] = *out;
  return MTD_OK;
}

// packed weights in the tile-major layout [rows/32][K/32][32][32] (mtd_conv_pack_*_blocked): rank-4 map
// (k_in = 32, n_in = 32, kstep = K/32, n_blk = rows/32), box (32, 32, 1, BN/32): a BN x 32 tile lands as BN rows of
// 128 B (SWIZZLE_128B) and is read from BN/32 contiguous 4 KB runs.
int make_w_map(CUtensorMap* out, const float* ptr, long long K, int rows, int BN) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return MTD_EINVAL;
  if (K % 32 || rows % 32 || BN % 32) return MTD_EINVAL;
  char keybuf[128];
  snprintf(keybuf, sizeof(keybuf), "W%p:%lld:%d:%d", (const void*)ptr, K, rows, BN);
  std::string key(keybuf);
  {
    std::lock_guard<std::mutex> lk(g_map_mutex);
    auto it = g_map_cache.find(key);
    if (it != g_map_cache.end()) { *out = it->second; return MTD_OK; }
  }
  const cuuint64_t KS = (cuuint64_t)(K / 32);
  cuuint64_t dims[4] = {32, 32, KS, (cuuint64_t)(rows / 32)};
  cuuint64_t strides[3] = {128, 4096, KS * 4096};
  cuuint32_t box[4] = {32, 32, 1, (cuuint32_t)(BN / 32)};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return MTD_EINVAL;
  std::lock_guard<std::mutex> lk(g_map_mutex);
  if (g_map_cache.size() > 8192) g_map_cache.clear();
  g_map_cache[key] = *out;
  return MTD_OK;
}

bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

// (H, W) = conv INPUT dims.  stride 1: size-preserving convs; stride 2: output (H+2p-k)/2+1 (the 4x4/pad-1 down* layers).
// The tile geometry is computed on the OUTPUT grid.
bool tc_geometry(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad, int* TW, int* TH, int* TB) {
  if (kh != kw || kh * kw > kMaxTaps) return false;
  if (stride == 1) { if (2 * pad != kh - 1) return false; }
  else if (stride == 2) {
    if ((H + 2 * pad - kh) % 2 || (W + 2 * pad - kw) % 2 || H + 2 * pad < kh || W + 2 * pad < kw) return false;
    H = (H + 2 * pad - kh) / 2 + 1; W = (W + 2 * pad - kw) / 2 + 1;
  } else return false;
  if (C1 <= 0 || C1 % 32 || C2 < 0 || C2 % 32 || N <= 0 || N % 32) return false;
  if (!is_pow2(W) || !is_pow2(H)) return false;
  if ((long long)B * H * W < 16) return false;
  int tw = W < kBM ? W : kBM;
  int th = kBM / tw;
  if (th > H) th = H;
  int tb = kBM / (tw * th);
  if (tw * th * tb != kBM || tb > 256) return false;
  *TW = tw; *TH = th; *TB = tb;
  return true;
}

template <int BN, int NPASS>
int launch_bn(const CUtensorMap& mA1, const CUtensorMap& mA2, const CUtensorMap& mB, const CUtensorMap& mBlo, TcArgs& a,
              cudaStream_t st) {
  const int stage_bytes = (NPASS == 3 ? 2 : 1) * (kABytes + BN * 128);
  int stages = (200 * 1024) / stage_bytes;
  if (stages > 6) stages = 6;
  a.stages = stages;
  size_t smem = 1024 + (size_t)stages * stage_bytes + 8 * (3 * stages + 4) + 16;
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BN, NPASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  mtd_launch(conv_tc_kernel<BN, NPASS>, a.grid, kThreads, smem, st, mA1, mA2, mB, mBlo, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// Tile width / work decomposition of the v1 kernel by a cost model (microseconds) fitted to the sweeps of
// tools/tune_tc.py over the layer shapes of the B = 20 train step (profiles/r01_tune_tc_*.txt):
//   T = F0 + waves * (Ft + K * ts[BN]) + [stream-K wave] * (Ft + per * ts[BN] + finish)
// F0 = launch + pipeline fill + drain, Ft = per-tile epilogue not hidden by the next tile, ts = one 32-channel k-step
// (L2 -> SM ingest of the A tile and the hi|lo weight tile, ~32 B/clk/SM), finish = the reduction launch reading the
// pieces of every stream-K tile from L2.  See "work decomposition" above WorkIter.
int g_tune_bn = 0, g_tune_per = 0;      // tools/tune_tc.py overrides: Cout tile; stream-K piece length (-1: none)

struct Schedule { int bn, n_dp, sk_tiles, sk_per, sk_P, grid; double cost; };

Schedule choose_schedule(int m_tiles, int N, int K, int passes, long long ws_floats, int n_align = 0) {
  const int sms = mtd_sm_count();
  Schedule best{};
  best.cost = 1e30;
  for (int bn = 128; bn >= 32; bn >>= 1) {
    if (N % bn) continue;
    if (n_align > 0 && n_align % bn) continue;        // split outputs: no tile may straddle the split
    if (g_tune_bn > 0 && bn != g_tune_bn && N % g_tune_bn == 0 && !(n_align > 0 && n_align % g_tune_bn)) continue;
    const double ts = (bn == 128 ? 0.78 : bn == 64 ? 0.57 : 0.52) * (passes == 3 ? 1.0 : 0.7);
    const double F0 = 6.0, Ft = 2.2;
    const int mn = m_tiles * (N / bn);
    // (a) whole tiles only
    if (g_tune_per <= 0) {
      const int waves = (mn + sms - 1) / sms;
      const double cost = F0 + waves * (Ft + K * ts);
      if (cost < best.cost) best = Schedule{bn, mn, 0, 0, 0, mn < sms ? mn : sms, cost};
    }
    // (b) full waves whole + the remainder as one stream-K wave
    const int n_dp = (mn / sms) * sms, rem = mn - n_dp;
    if (rem == 0 || ws_floats <= 0 || g_tune_per < 0) continue;
    const long long total = (long long)rem * K;
    const int per_min = (int)((total + sms - 1) / sms);
    for (int f = 0; f < 8; ++f) {
      static const double mult[8] = {1.0, 1.25, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0};
      int per = g_tune_per > 0 ? g_tune_per : (int)(per_min * mult[f] + 0.5);
      if (per < per_min) per = per_min;
      if (per < 2 && K >= 2) per = 2;
      if (per >= K && n_dp == 0 && g_tune_per <= 0) break;     // no split left: covered by (a)
      const int grid_sk = (int)((total + per - 1) / per);
      const int P = (K - 1) / per + 2;
      if ((long long)rem * P * kBM * bn > ws_floats) continue;
      const double pieces = (double)K / per + 1.0;                       // average pieces per stream-K tile
      const double fin = 3.0 + (double)rem * kBM * bn * 4.0 * (pieces + 1.0) / 2.5e6;     // L2-resident traffic at ~2.5 TB/s
      const double per_cta_pieces = (double)per / K + 1.0;
      const double cost = F0 + (n_dp / sms) * (Ft + K * ts) + per_cta_pieces * Ft + per * ts + fin;
      if (cost < best.cost) best = Schedule{bn, n_dp, rem, per, P, n_dp ? sms : grid_sk, cost};
      if (g_tune_per > 0) break;
    }
  }
  return best;
}

// ---- v2 host side -------------------------------------------------------------------------------------
int g_tc_version = 1;      // 1 (default): A through shared memory (conv_tc_kernel); 2: A through TMEM, MT pixel tiles per CTA
                           // (slower on every measured layer shape -- kept selectable for experiments, see DESIGN.md)

struct V2Cfg { int bn, mt; };
constexpr V2Cfg kV2Cfgs[3] = {{128, 3}, {64, 6}, {32, 8}};

void choose_tiling_v2(int m_tiles, int N, int kiters, int passes, int force_split, int* cfg_out, int* ksplit_out) {
  const int sms = mtd_sm_count();
  double best = 1e30;
  int bc = -1, bks = 1;
  for (int ci = 0; ci < 3; ++ci) {
    const int bn = kV2Cfgs[ci].bn, mt = kV2Cfgs[ci].mt;
    if (N % bn) continue;
    const int groups = (m_tiles + mt - 1) / mt;
    const double mtv = (double)m_tiles / groups;                      // average pixel tiles per group
    const int mn = groups * (N / bn);
    const double mma = mtv * (passes == 3 ? 12.0 : 4.0) * (bn / 2.0);  // cycles: 4 k-slices x passes, 128 x bn x 8 each
    const double byt = (mtv * 16.0 + (passes == 3 ? 2.0 : 1.0) * bn / 8.0) * 1024.0 / 36.0;
    double t_step = mma > byt ? mma : byt;
    if (t_step < 1200.0) t_step = 1200.0;
    int ks = 1;
    if (force_split > 0) ks = force_split;
    else if (mn < sms && kiters >= 8) {
      ks = sms / mn;
      if (ks > kiters / 2) ks = kiters / 2;
      if (ks < 1) ks = 1;
    }
    const int kper = (kiters + ks - 1) / ks;
    ks = (kiters + kper - 1) / kper;
    const int rounds = (mn * ks + sms - 1) / sms;
    const double cost = (double)rounds * (kper * t_step + mtv * bn * 24.0 + 4000.0) + (ks > 1 ? 8000.0 : 0.0);
    if (cost < best) { best = cost; bc = ci; bks = ks; }
  }
  *cfg_out = bc;
  *ksplit_out = bks;
}

template <int BN, int MT, int NPASS>
int launch_v2(const CUtensorMap& mA1, const CUtensorMap& mA2, const CUtensorMap& mB, const CUtensorMap& mBlo, TcArgs& a,
              cudaStream_t st) {
  const int b_bytes = (NPASS == 3 ? 2 : 1) * BN * 128;
  a.rb = 2;
  int ra = (200 * 1024 - a.rb * b_bytes) / kABytes;
  if (ra > 10) ra = 10;
  a.ra = ra;
  size_t smem = 1024 + (size_t)a.ra * kABytes + (size_t)a.rb * b_bytes + 8 * (2 * a.ra + 2 * a.rb + 8);
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(conv_tc2_kernel<BN, MT, NPASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  int grid = a.n_tiles < mtd_sm_count() ? a.n_tiles : mtd_sm_count();
  mtd_launch(conv_tc2_kernel<BN, MT, NPASS>, grid, kThreads, smem, st, mA1, mA2, mB, mBlo, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// v1 kernel: whole-tile waves + one stream-K wave (choose_schedule), partial sums through a.ws, no atomics.
int launch_tc_v1(const float* x1, const float* x2, const float* wp, int passes, TcArgs& a, cudaStream_t st) {
  const int m_tiles = a.n_wt * a.n_ht * a.n_bt;
  const int kiters = a.T * (a.kc1 + a.kc2);
  if (a.ws && !mtd_aligned16(a.ws)) return MTD_EALIGN;
  if (a.n_cls < 1) a.n_cls = 1;
  const Schedule sc = choose_schedule(m_tiles * a.n_cls, a.N, kiters, passes, a.ws ? a.ws_floats : 0, a.n_split);
  if (sc.cost >= 1e30) return MTD_EINVAL;
  const int BN = sc.bn;
  a.n_nt = a.N / BN;
  a.tiles_per_cls = m_tiles * a.n_nt;
  a.n_tiles = a.tiles_per_cls * a.n_cls;
  a.n_dp = sc.n_dp; a.sk_tiles = sc.sk_tiles; a.sk_per = sc.sk_per; a.sk_P = sc.sk_P; a.grid = sc.grid;
  a.ksplit = 1; a.kper = kiters;
  CUtensorMap mA1, mA2, mB;
  if (a.es < 1) { a.es = 1; a.inH = a.H; a.inW = a.W; }
  int rc = make_act_map(&mA1, x1, a.C1, a.inW, a.inH, a.B, a.TW, a.TH, a.TB, false, a.es);
  if (rc) return rc;
  if (a.C2) { rc = make_act_map(&mA2, x2, a.C2, a.inW, a.inH, a.B, a.TW, a.TH, a.TB, false, a.es); if (rc) return rc; }
  else mA2 = mA1;
  const long long K = (long long)a.T * (a.C1 + a.C2);
  rc = make_w_map(&mB, wp, K, a.N * a.n_cls, BN);
  if (rc) return rc;
  CUtensorMap mBlo = mB;
  if (passes == 3) {
    // the lo half follows the hi half of the FULL packed weight (a.wrows_total rows), not of this row slice
    rc = make_w_map(&mBlo, wp + (size_t)a.wrows_total * K, K, a.N * a.n_cls, BN);
    if (rc) return rc;
  }
#define TC_DISPATCH(BN_)                                                           \
  rc = passes == 3 ? launch_bn<BN_, 3>(mA1, mA2, mB, mBlo, a, st) : launch_bn<BN_, 1>(mA1, mA2, mB, mBlo, a, st)
  if (BN == 128) { TC_DISPATCH(128); }
  else if (BN == 64) { TC_DISPATCH(64); }
  else { TC_DISPATCH(32); }
#undef TC_DISPATCH
  if (rc) return rc;
  if (a.sk_tiles > 0) {
    const long long work = (long long)a.sk_tiles * kBM * (BN / 4);
    int blocks = (int)((work + 255) / 256);
    if (blocks > mtd_sm_count() * 8) blocks = mtd_sm_count() * 8;
    mtd_launch(tc_sk_finish_kernel, blocks, 256, 0, st, a, BN, kiters);
    MTD_CHECK_LAUNCH();
  }
  return MTD_OK;
}

int g_c32_enabled = 1;      // mtd_tc_set_c32(0) routes 32 -> 32 3x3 layers through the general kernel (A/B measurements)

bool c32_eligible(const TcArgs& a) {
  if (!g_c32_enabled || g_tc_version != 1) return false;
  if (a.C1 != 32 || a.C2 != 0 || a.N != 32 || a.T != 9 || a.es > 1 || a.n_cls > 1 || a.n_split != 0) return false;
  if (a.omy != 1 || a.omx != 1 || a.ooy != 0 || a.oox != 0 || a.outH != a.H || a.outW != a.W) return false;
  if (a.H % 16 || a.W % 8) return false;
  bool seen[9] = {};
  for (int t = 0; t < 9; ++t) {       // the taps must be exactly the 3 x 3 neighbourhood (any order)
    if (a.dy[t] < -1 || a.dy[t] > 1 || a.dx[t] < -1 || a.dx[t] > 1) return false;
    seen[(a.dy[t] + 1) * 3 + a.dx[t] + 1] = true;
  }
  for (bool s_ : seen) if (!s_) return false;
  return true;
}

template <int NPASS>
int launch_c32_n(const CUtensorMap& mA, const CUtensorMap& mB, const CUtensorMap& mBlo, TcArgs& a, cudaStream_t st) {
  const size_t smem = 1024 + kC32WBytes + 2 * kRawStage + 2 * kCvStage + 8 * 14 + 16;
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(conv_c32_kernel<NPASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  mtd_launch(conv_c32_kernel<NPASS>, a.grid, kThreads, smem, st, mA, mB, mBlo, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int launch_c32(const float* x, const float* wp, int passes, TcArgs& a, cudaStream_t st) {
  a.n_wt = a.W / 8; a.n_ht = a.H / 16;
  a.n_tiles = a.B * a.n_wt * a.n_ht;
  a.grid = a.n_tiles < mtd_sm_count() ? a.n_tiles : mtd_sm_count();
  CUtensorMap mA, mB;
  int rc = make_act_map(&mA, x, 32, a.W, a.H, a.B, kHaloW, kHaloH, 1, false, 1);
  if (rc) return rc;
  const long long K = 9 * 32;
  rc = make_w_map(&mB, wp, K, 32, 32);
  if (rc) return rc;
  CUtensorMap mBlo = mB;
  if (passes == 3) {
    rc = make_w_map(&mBlo, wp + (size_t)a.wrows_total * K, K, 32, 32);
    if (rc) return rc;
  }
  return passes == 3 ? launch_c32_n<3>(mA, mB, mBlo, a, st) : launch_c32_n<1>(mA, mB, mBlo, a, st);
}

// ---- general halo-tile kernel (3x3 / stride 1, C and N multiples of 32): host side ------------------------------------
int g_halo_enabled = 1;     // mtd_tc_set_halo(0) routes these layers through the tap-streaming kernel (A/B measurements)

bool taps_are_3x3(const TcArgs& a) {
  if (a.T != 9) return false;
  bool seen[9] = {};
  for (int t = 0; t < 9; ++t) {       // exactly the 3 x 3 neighbourhood (any order)
    if (a.dy[t] < -1 || a.dy[t] > 1 || a.dx[t] < -1 || a.dx[t] > 1) return false;
    seen[(a.dy[t] + 1) * 3 + a.dx[t] + 1] = true;
  }
  for (bool s_ : seen) if (!s_) return false;
  return true;
}

bool halo_eligible(const TcArgs& a) {
  if (!g_halo_enabled || g_tc_version != 1) return false;
  if (a.C1 % 32 || a.C2 % 32 || a.N % 32 || a.es > 1 || a.n_cls > 1) return false;
  if (a.omy != 1 || a.omx != 1 || a.ooy != 0 || a.oox != 0 || a.outH != a.H || a.outW != a.W) return false;
  if (a.H % 16 || a.W % 8) return false;
  return taps_are_3x3(a);
}

template <int BN, int NPASS>
int launch_halo_bn(const CUtensorMap& mA1, const CUtensorMap& mA2, const CUtensorMap& mB, const CUtensorMap& mBlo, TcArgs& a,
                   cudaStream_t st) {
  constexpr int kBStage = (NPASS == 3 ? 2 : 1) * BN * 128;
  const int avail = 227 * 1024 - 1024 - 512 - 2 * kCvStage;
  a.ra = (avail - 2 * kRawStage) / kBStage >= 3 ? 2 : 1;          // two raw halo stages unless that starves the weight ring
  int stages = (avail - a.ra * kRawStage) / kBStage;
  if (stages > 6) stages = 6;
  if (stages < 2) return MTD_EINVAL;
  a.stages = stages;
  const size_t smem = 1024 + (size_t)a.ra * kRawStage + 2 * kCvStage + (size_t)stages * kBStage + 8 * (13 + 2 * stages) + 16;
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(conv_halo_kernel<BN, NPASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  mtd_launch(conv_halo_kernel<BN, NPASS>, a.grid, kThreads, smem, st, mA1, mA2, mB, mBlo, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int launch_halo(const float* x1, const float* x2, const float* wp, int passes, TcArgs& a, cudaStream_t st) {
  a.TW = 8; a.TH = 16; a.TB = 1;
  a.n_wt = a.W / 8; a.n_ht = a.H / 16; a.n_bt = a.B;
  const int m_tiles = a.n_wt * a.n_ht * a.n_bt;
  a.m_tiles = m_tiles;
  a.kc1 = a.C1 / 32; a.kc2 = a.C2 / 32;
  const int kiters = 9 * (a.kc1 + a.kc2);
  if (a.ws && !mtd_aligned16(a.ws)) return MTD_EALIGN;
  a.n_cls = 1;
  const Schedule sc = choose_schedule(m_tiles, a.N, kiters, passes, a.ws ? a.ws_floats : 0, a.n_split);
  if (sc.cost >= 1e30) return MTD_EINVAL;
  const int BN = sc.bn;
  a.n_nt = a.N / BN;
  a.tiles_per_cls = m_tiles * a.n_nt;
  a.n_tiles = a.tiles_per_cls;
  a.n_dp = sc.n_dp; a.sk_tiles = sc.sk_tiles; a.sk_per = sc.sk_per; a.sk_P = sc.sk_P; a.grid = sc.grid;
  a.ksplit = 1; a.kper = kiters;
  a.es = 1; a.inH = a.H; a.inW = a.W;
  CUtensorMap mA1, mA2, mB;
  int rc = make_act_map(&mA1, x1, a.C1, a.W, a.H, a.B, kHaloW, kHaloH, 1, false, 1);
  if (rc) return rc;
  if (a.C2) { rc = make_act_map(&mA2, x2, a.C2, a.W, a.H, a.B, kHaloW, kHaloH, 1, false, 1); if (rc) return rc; }
  else mA2 = mA1;
  const long long K = 9LL * (a.C1 + a.C2);
  rc = make_w_map(&mB, wp, K, a.N, BN);
  if (rc) return rc;
  CUtensorMap mBlo = mB;
  if (passes == 3) {
    rc = make_w_map(&mBlo, wp + (size_t)a.wrows_total * K, K, a.N, BN);
    if (rc) return rc;
  }
#define HALO_DISPATCH(BN_)                                                                \
  rc = passes == 3 ? launch_halo_bn<BN_, 3>(mA1, mA2, mB, mBlo, a, st) : launch_halo_bn<BN_, 1>(mA1, mA2, mB, mBlo, a, st)
  if (BN == 128) { HALO_DISPATCH(128); }
  else if (BN == 64) { HALO_DISPATCH(64); }
  else { HALO_DISPATCH(32); }
#undef HALO_DISPATCH
  if (rc) return rc;
  if (a.sk_tiles > 0) {
    const long long work = (long long)a.sk_tiles * kBM * (BN / 4);
    int blocks = (int)((work + 255) / 256);
    if (blocks > mtd_sm_count() * 8) blocks = mtd_sm_count() * 8;
    mtd_launch(tc_sk_finish_kernel, blocks, 256, 0, st, a, BN, kiters);
    MTD_CHECK_LAUNCH();
  }
  return MTD_OK;
}

// wp: packed weights, tile-major (mtd_conv_pack_*_blocked); for passes == 3 the buffer holds [hi | lo].
// v2 kernel only: `finish` = run the split-K finishing pass here (false when the caller batches several launches into
// one output, e.g. the four parity classes of a stride-2 dgrad); the chosen ksplit is returned through a.ksplit.
int launch_tc(const float* x1, const float* x2, const float* wp, int passes, TcArgs& a, cudaStream_t st, int force_split = 0,
              bool finish = true) {
  if (passes != 1 && passes != 3) return MTD_EINVAL;
  if (!tc_geometry(a.B, a.H, a.W, a.C1, a.C2, a.N, 1, 1, 1, 0, &a.TW, &a.TH, &a.TB)) return MTD_EINVAL;
  if (!mtd_aligned16(x1) || !mtd_aligned16(wp) || !mtd_aligned16(a.out) || (x2 && !mtd_aligned16(x2)) ||
      (a.bias && !mtd_aligned16(a.bias)))
    return MTD_EALIGN;
  if (c32_eligible(a)) return launch_c32(x1, wp, passes, a, st);
  if (halo_eligible(a)) return launch_halo(x1, x2, wp, passes, a, st);
  a.n_wt = a.W / a.TW; a.n_ht = a.H / a.TH; a.n_bt = (a.B + a.TB - 1) / a.TB;
  const int m_tiles = a.n_wt * a.n_ht * a.n_bt;
  a.kc1 = a.C1 / 32; a.kc2 = a.C2 / 32;
  a.m_tiles = m_tiles;
  if (g_tc_version != 2) return launch_tc_v1(x1, x2, wp, passes, a, st);
  const int kiters = a.T * (a.kc1 + a.kc2);
  const int sms = mtd_sm_count();
  int BN = 32, ksplit = 1, v2cfg = -1;
  choose_tiling_v2(m_tiles, a.N, kiters, passes, force_split, &v2cfg, &ksplit);
  if (v2cfg < 0) return MTD_EINVAL;
  BN = kV2Cfgs[v2cfg].bn;
  a.n_groups = (m_tiles + kV2Cfgs[v2cfg].mt - 1) / kV2Cfgs[v2cfg].mt;
  a.n_nt = a.N / BN;
  int mn_tiles = a.n_groups * a.n_nt;
  a.kper = (kiters + ksplit - 1) / ksplit;
  ksplit = (kiters + a.kper - 1) / a.kper;          // no empty splits
  a.ksplit = ksplit;
  a.n_tiles = mn_tiles * ksplit;
  const size_t total = (size_t)a.B * a.outH * a.outW * a.N;
  if (ksplit > 1 && finish) MTD_CUDA(cudaMemsetAsync(a.out, 0, total * sizeof(float), st));
  CUtensorMap mA1, mA2, mB;
  if (a.es < 1) { a.es = 1; a.inH = a.H; a.inW = a.W; }
  int rc = make_act_map(&mA1, x1, a.C1, a.inW, a.inH, a.B, a.TW, a.TH, a.TB, false, a.es);
  if (rc) return rc;
  if (a.C2) { rc = make_act_map(&mA2, x2, a.C2, a.inW, a.inH, a.B, a.TW, a.TH, a.TB, false, a.es); if (rc) return rc; }
  else mA2 = mA1;
  const long long K = (long long)a.T * (a.C1 + a.C2);
  rc = make_w_map(&mB, wp, K, a.N, BN);
  if (rc) return rc;
  CUtensorMap mBlo = mB;
  if (passes == 3) {
    rc = make_w_map(&mBlo, wp + (size_t)a.wrows_total * K, K, a.N, BN);
    if (rc) return rc;
  }
#define TC2_DISPATCH(BN_, MT_)                                                     \
  rc = passes == 3 ? launch_v2<BN_, MT_, 3>(mA1, mA2, mB, mBlo, a, st) : launch_v2<BN_, MT_, 1>(mA1, mA2, mB, mBlo, a, st)
  if (v2cfg == 0) { TC2_DISPATCH(128, 3); }
  else if (v2cfg == 1) { TC2_DISPATCH(64, 6); }
  else { TC2_DISPATCH(32, 8); }
#undef TC2_DISPATCH
  if (rc) return rc;
  if (ksplit > 1 && finish) {
    int blocks = (int)((total + 255) / 256);
    if (blocks > sms * 8) blocks = sms * 8;
    mtd_launch(tc_finish_kernel, blocks, 256, 0, st, a, total);
    MTD_CHECK_LAUNCH();
  }
  return MTD_OK;
}

__global__ void split_tf32_kernel(float* __restrict__ hi, float* __restrict__ lo, size_t n) {
  mtd_pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float w = hi[i];
    uint32_t h, l;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(w));
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(w - __uint_as_float(h)));
    hi[i] = __uint_as_float(h);
    lo[i] = __uint_as_float(l);
  }
}


// =====================================================================================================
// Weight gradient on the tensor cores.
//
//   gp[n][t][c] = sum_p dz[p][n] * x[p@t][c]          (p = output pixel, x[p@t] = input pixel of tap t)
//
// GEMM with K = pixels.  Both operands have the reduction (pixel) dimension as their SLOW memory dimension
// (NHWC), i.e. they are MN-major: a TMA box (32 channels, Kp pixels) lands as Kp rows of 128 B, which (with the
// 128B_ATOM_32B swizzle) is the canonical MN-major SW128_32B atom stack (4 pixel rows = one 512 B k-atom;
// 32 channels = one mn-block).
//   A (M side, 128 rows) = 4 mn-blocks: "units" u = t*kchunks + cc (tap t, 32-channel chunk cc) 4j..4j+3,
//                          each the tap-shifted box of x — for C = 32 layers one MMA covers 4 taps at once
//   B (N side, BN cols)  = BN/32 mn-blocks of the dz box (unshifted)
// so D[row = (unit, ch)][col = n] accumulates in TMEM over the CTA's share of the pixel tiles (split-K over
// pixels), and the epilogue atomically adds the fp32 partials into the packed gradient.  Both operands are
// activations, so the rounding warps split BOTH into tf32 hi/lo for the 3xTF32 mode.
// =====================================================================================================
// KP = pixels per k-step (32 for the 3xTF32 mode, 64 for plain TF32); one (32 ch x KP px) block = KP * 128 bytes

struct WgArgs {
  int B, H, W, C1, C2, N, T;
  int dy[kMaxTaps], dx[kMaxTaps];
  int TW, TH, TB, n_wt, n_ht, n_bt;            // pixel-tile geometry over the OUTPUT grid (TW*TH*TB == KP)
  int es;                                       // conv stride: x boxes are loaded with elementStrides es
  int kc1, kc2, units, m_tiles, n_nt;
  int ksplit, kper, ptiles, n_tiles, stages;
  float* gp;
};

__host__ __device__ constexpr uint32_t make_idesc_mn(int bn) {      // both operands MN-major
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(bn >> 3) << 17) |
         ((uint32_t)(kBM >> 4) << 24);
}
// MN-major descriptor.  For 32-bit (tf32) MN-major operands the ONLY layout the tensor core accepts is
// SWIZZLE_128B_BASE32B (layout type 1; cutlass sm100_common.inl: "for mn-major tf32 operands, SW128_32B is the
// only available smem layout"): Swizzle<2,5,2>, atom = 32 channels (128 B) x 4 pixel rows, produced by TMA's
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.  LBO = byte stride between 32-channel mn-blocks, SBO = 512 B between
// 4-pixel k-atoms (one K = 8 MMA spans two of them).
__device__ __forceinline__ uint64_t make_sw128_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | (32ull << 32) | (1ull << 46) | (1ull << 61);
}

template <int BN, int NPASS, int KP>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapX1, const __grid_constant__ CUtensorMap mapX2,
                const __grid_constant__ CUtensorMap mapDz, const __grid_constant__ WgArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kBlkBytes = KP * 128;
  constexpr int kNB = BN / 32;                                  // dz blocks
  constexpr int kBlocks = 4 + kNB;                              // fp32 blocks landed by TMA per stage
  constexpr int kHalf = kBlocks * kBlkBytes;                    // hi tiles (in place); lo tiles follow
  constexpr int kStageBytes = (NPASS == 3 ? 2 : 1) * kHalf;
  constexpr uint32_t kTmemCols = (2 * BN) < 32 ? 32 : 2 * BN;

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int S = a.stages;
  const uint32_t bar_base = base + (uint32_t)S * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
  auto conv_bar = [&](int s) { return bar_base + 8u * (2 * S + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (3 * S + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (3 * S + 2 + i); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * S + 4);
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.kc1 + a.kc2;
  const int Ctot = kchunks * 32;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapX1);
    if (a.kc2) prefetch_tmap(&mapX2);
    prefetch_tmap(&mapDz);
    for (int s = 0; s < S; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      mbar_init(conv_bar(s), 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  // barriers initialised, TMEM allocated, descriptors prefetched: all of it overlapped the previous kernel's tail
  mtd_pdl_prologue();

  // tile = ((mt * n_nt) + nt) * ksplit + ks
  auto decode_tile = [&](int tile, int& mt, int& n0, int& k_begin, int& k_end) {
    const int ks = tile % a.ksplit;
    tile /= a.ksplit;
    k_begin = ks * a.kper;
    k_end = min(a.ptiles, k_begin + a.kper);
    n0 = (tile % a.n_nt) * BN;
    mt = tile / a.n_nt;
  };
  auto decode_ptile = [&](int pt, int& b0, int& h0, int& w0) {
    int mw = pt % a.n_wt;
    pt /= a.n_wt;
    int mh = pt % a.n_ht, mb = pt / a.n_ht;
    b0 = mb * a.TB; h0 = mh * a.TH; w0 = mw * a.TW;
  };

  if (warp == 0) {
    if (lane == 0) {
      PipeState st;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int mt, n0, k_begin, k_end;
        decode_tile(tile, mt, n0, k_begin, k_end);
        int nvalid = min(4, a.units - mt * 4);
        for (int it = k_begin; it < k_end; ++it) {
          int b0, h0, w0;
          decode_ptile(it, b0, h0, w0);
          mbar_wait(empty_bar(st.stage), st.phase ^ 1u);
          mbar_expect_tx(full_bar(st.stage), (uint32_t)(nvalid + kNB) * kBlkBytes);
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes;
          for (int i = 0; i < nvalid; ++i) {
            const int u = mt * 4 + i, t = u / kchunks, cc = u - t * kchunks;
            if (cc < a.kc1) tma_load_4d(&mapX1, sa + i * kBlkBytes, full_bar(st.stage), cc * 32, w0 * a.es + a.dx[t], h0 * a.es + a.dy[t], b0);
            else tma_load_4d(&mapX2, sa + i * kBlkBytes, full_bar(st.stage), (cc - a.kc1) * 32, w0 * a.es + a.dx[t], h0 * a.es + a.dy[t], b0);
          }
#pragma unroll
          for (int j = 0; j < kNB; ++j)
            tma_load_4d(&mapDz, sa + (4 + j) * kBlkBytes, full_bar(st.stage), n0 + j * 32, w0, h0, b0);
          st.advance(S);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState st;
      constexpr uint32_t idesc = make_idesc_mn(BN);
      int lt = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
        int mt, n0, k_begin, k_end;
        decode_tile(tile, mt, n0, k_begin, k_end);
        const int acc = lt & 1;
        const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int it = k_begin; it < k_end; ++it) {
          mbar_wait(conv_bar(st.stage), st.phase);
          tc_fence_after();
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes;
          const uint64_t da = make_sw128_desc_mn(sa, kBlkBytes), db = make_sw128_desc_mn(sa + 4 * kBlkBytes, kBlkBytes);
#pragma unroll
          for (int kk = 0; kk < KP / 8; ++kk) {       // one 8-pixel k-atom (1024 B) per MMA: +64 in 16-byte units
            const uint32_t accum = (it > k_begin || kk > 0) ? 1u : 0u;
            if (NPASS == 3) {
              const uint64_t dal = make_sw128_desc_mn(sa + kHalf, kBlkBytes), dbl = make_sw128_desc_mn(sa + kHalf + 4 * kBlkBytes, kBlkBytes);
              umma_tf32(tmem_d, dal + 64u * kk, db + 64u * kk, idesc, accum);
              umma_tf32(tmem_d, da + 64u * kk, dbl + 64u * kk, idesc, 1u);
              umma_tf32(tmem_d, da + 64u * kk, db + 64u * kk, idesc, 1u);
            } else {
              umma_tf32(tmem_d, da + 64u * kk, db + 64u * kk, idesc, accum);
            }
          }
          umma_commit(empty_bar(st.stage));
          st.advance(S);
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else if (warp < 6) {
    const int ct = threadIdx.x - 64;
    PipeState st;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      int mt, n0, k_begin, k_end;
      decode_tile(tile, mt, n0, k_begin, k_end);
      for (int it = k_begin; it < k_end; ++it) {
        mbar_wait(full_bar(st.stage), st.phase);
        float4* tileA = reinterpret_cast<float4*>(gen_base + (size_t)st.stage * kStageBytes);
#pragma unroll 4
        for (int j = 0; j < kHalf / 16 / 128; ++j) {
          float4 v = tileA[ct + 128 * j];
          uint32_t r0, r1, r2, r3;
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r0) : "f"(v.x));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r1) : "f"(v.y));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r2) : "f"(v.z));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r3) : "f"(v.w));
          const float4 hi = make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float(r2), __uint_as_float(r3));
          tileA[ct + 128 * j] = hi;
          if (NPASS == 3) {
            uint32_t l0, l1, l2, l3;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l0) : "f"(v.x - hi.x));
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l1) : "f"(v.y - hi.y));
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l2) : "f"(v.z - hi.z));
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l3) : "f"(v.w - hi.w));
            tileA[kHalf / 16 + ct + 128 * j] =
                make_float4(__uint_as_float(l0), __uint_as_float(l1), __uint_as_float(l2), __uint_as_float(l3));
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(conv_bar(st.stage));
        st.advance(S);
      }
    }
  } else {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    int lt = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
      int mt, n0, k_begin, k_end;
      decode_tile(tile, mt, n0, k_begin, k_end);
      const int acc = lt & 1;
      const uint32_t acc_phase = (uint32_t)(lt >> 1) & 1u;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int u = mt * 4 + (r >> 5);
      const bool valid = u < a.units;
      const int t = valid ? u / kchunks : 0, cc = valid ? u - t * kchunks : 0;
      const int c = cc * 32 + (r & 31);
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c0), v);
        if (valid) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float* dst = a.gp + ((size_t)(n0 + c0 + j) * a.T + t) * Ctot + c;
            if (a.ksplit > 1) atomicAdd(dst, __uint_as_float(v[j]));
            else *dst = __uint_as_float(v[j]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

template <int BN, int NPASS, int KP>
int launch_wg(const CUtensorMap& mX1, const CUtensorMap& mX2, const CUtensorMap& mDz, WgArgs& a, cudaStream_t st) {
  const int stage_bytes = (NPASS == 3 ? 2 : 1) * (4 + BN / 32) * KP * 128;
  int stages = (200 * 1024) / stage_bytes;
  if (stages > 8) stages = 8;
  if (stages > a.kper) stages = a.kper < 2 ? 2 : a.kper;
  a.stages = stages;
  size_t smem = 1024 + (size_t)stages * stage_bytes + 8 * (3 * stages + 4) + 16;
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<BN, NPASS, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  int grid = a.n_tiles < mtd_sm_count() ? a.n_tiles : mtd_sm_count();
  mtd_launch(wgrad_tc_kernel<BN, NPASS, KP>, grid, kThreads, smem, st, mX1, mX2, mDz, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

bool wg_geometry(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad, int kKp, int* TW, int* TH, int* TB) {
  if (kh != kw || kh * kw > kMaxTaps) return false;
  if (stride == 1) { if (2 * pad != kh - 1) return false; }
  else if (stride == 2) {
    if ((H + 2 * pad - kh) % 2 || (W + 2 * pad - kw) % 2 || H + 2 * pad < kh || W + 2 * pad < kw) return false;
    H = (H + 2 * pad - kh) / 2 + 1; W = (W + 2 * pad - kw) / 2 + 1;
  } else return false;
  if (C1 <= 0 || C1 % 32 || C2 < 0 || C2 % 32 || N <= 0 || N % 32) return false;
  if (!is_pow2(W) || !is_pow2(H)) return false;
  int tw = W < kKp ? W : kKp;
  int th = kKp / tw;
  if (th > H) th = H;
  int tb = kKp / (tw * th);
  if (tw * th * tb != kKp) return false;
  *TW = tw; *TH = th; *TB = tb;
  return true;
}

// ---- weight gradient of a 3x3 / stride-1 / pad-1 layer with an output grid of at least 8 x 8, plain TF32 -----------
// The tap-streaming kernel above lands every x pixel 9 times (once per tap) per Cout tile, and dz once per 4 units.
// Here a k-step is one 8 x 8 pixel tile of one image, and a CTA tile is (32-channel chunk cc, BN dz channels, pixel
// range): per k-step the producer lands three dx-shifted HALO boxes of x — 10 rows x 8 columns, image rows h0-1 .. h0+8,
// columns w0+dx .. w0+dx+7, zero outside the image — and the BN/32 dz blocks, once for all 9 taps.
// In the MN-major SW128_32B layout a pixel is one 128 B row, so a box row of 8 pixels is 1024 B: a whole number of
// swizzle repeats, like the 1024 B k-atom steps (+64 in 16 B units) that every MN-major MMA here already takes.  The dy
// shift is therefore a pure start-address offset, and the M = 128 operand whose four mn-blocks lie LBO = 1024 B apart is
// the dx box seen at dy = -1, 0, +1 (+2 is a fourth, unused shift: its rows read the next 1 KB of the stage, which is
// always landed data, and are never stored).  Three accumulators (dx = -1, 0, +1) of BN columns each.
// L2 -> SM bytes per k-step: 3 x 10 KB + BN x 256 B for 9 x 32 x BN outputs, against (4 + BN/32) x 8 KB for 4 x 32 x BN
// on the tap-streaming kernel: 2.3x (BN = 128) to 3.2x (BN = 32) fewer bytes per FLOP.
constexpr int kHaloPx = 8;                                  // pixel tile edge
constexpr int kHaloBoxBytes = kHaloPx * (kHaloPx + 2) * 128;  // one dx box: 10 rows x 8 pixels x 32 channels

__host__ __device__ constexpr int wgh_stage_bytes(int bn) { return 3 * kHaloBoxBytes + (bn / 32) * 64 * 128; }
__host__ __device__ constexpr int wgh_acc_bufs(int bn) { return 6 * bn <= 512 ? 2 : 1; }    // double-buffered if it fits

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap mapX1, const __grid_constant__ CUtensorMap mapX2,
                  const __grid_constant__ CUtensorMap mapDz, const __grid_constant__ WgArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int kBlkBytes = 64 * 128;                           // one 32-channel dz block of the 64-pixel tile
  constexpr int kNB = BN / 32;
  constexpr int kStageBytes = wgh_stage_bytes(BN);
  constexpr int kNAcc = wgh_acc_bufs(BN);
  constexpr uint32_t kAccCols = 3 * BN;
  constexpr uint32_t kTmemCols = kNAcc * kAccCols <= 256 ? 256 : 512;

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int S = a.stages;
  const uint32_t bar_base = base + (uint32_t)S * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
  auto conv_bar = [&](int s) { return bar_base + 8u * (2 * S + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (3 * S + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (3 * S + 2 + i); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * S + 4);
  unsigned char* gen_base = smem_raw + (base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.kc1 + a.kc2;
  const int Ctot = kchunks * 32;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapX1);
    if (a.kc2) prefetch_tmap(&mapX2);
    prefetch_tmap(&mapDz);
    for (int s = 0; s < S; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      mbar_init(conv_bar(s), 4);
    }
    for (int i = 0; i < kNAcc; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - base));
  mtd_pdl_prologue();

  // tile = ((cc * n_nt) + nt) * ksplit + ks
  auto decode_tile = [&](int tile, int& cc, int& n0, int& k_begin, int& k_end) {
    const int ks = tile % a.ksplit;
    tile /= a.ksplit;
    k_begin = ks * a.kper;
    k_end = min(a.ptiles, k_begin + a.kper);
    n0 = (tile % a.n_nt) * BN;
    cc = tile / a.n_nt;
  };

  if (warp == 0) {
    if (lane == 0) {
      PipeState st;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int cc, n0, k_begin, k_end;
        decode_tile(tile, cc, n0, k_begin, k_end);
        const CUtensorMap* mx = cc < a.kc1 ? &mapX1 : &mapX2;
        const int c0 = (cc < a.kc1 ? cc : cc - a.kc1) * 32;
        for (int it = k_begin; it < k_end; ++it) {
          int pt = it;
          const int w0 = (pt % a.n_wt) * kHaloPx;
          pt /= a.n_wt;
          const int h0 = (pt % a.n_ht) * kHaloPx, b0 = pt / a.n_ht;
          mbar_wait(empty_bar(st.stage), st.phase ^ 1u);
          mbar_expect_tx(full_bar(st.stage), (uint32_t)kStageBytes);
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes;
#pragma unroll
          for (int i = 0; i < 3; ++i) tma_load_4d(mx, sa + i * kHaloBoxBytes, full_bar(st.stage), c0, w0 + i - 1, h0 - 1, b0);
#pragma unroll
          for (int j = 0; j < kNB; ++j)
            tma_load_4d(&mapDz, sa + 3 * kHaloBoxBytes + j * kBlkBytes, full_bar(st.stage), n0 + j * 32, w0, h0, b0);
          st.advance(S);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState st;
      constexpr uint32_t idesc = make_idesc_mn(BN);
      int lt = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
        int cc, n0, k_begin, k_end;
        decode_tile(tile, cc, n0, k_begin, k_end);
        const int acc = lt % kNAcc;
        const uint32_t acc_phase = (uint32_t)(lt / kNAcc) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * kAccCols);
        for (int it = k_begin; it < k_end; ++it) {
          mbar_wait(conv_bar(st.stage), st.phase);
          tc_fence_after();
          const uint32_t sa = base + (uint32_t)st.stage * kStageBytes;
          const uint64_t db = make_sw128_desc_mn(sa + 3 * kHaloBoxBytes, kBlkBytes);
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const uint64_t da = make_sw128_desc_mn(sa + i * kHaloBoxBytes, kHaloPx * 128);     // mn-block j = dy + 1
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
              umma_tf32(tmem_d + i * BN, da + 64u * kk, db + 64u * kk, idesc, (it > k_begin || kk > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(st.stage));
          st.advance(S);
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else if (warp < 6) {
    const int ct = threadIdx.x - 64;
    PipeState st;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      int cc, n0, k_begin, k_end;
      decode_tile(tile, cc, n0, k_begin, k_end);
      for (int it = k_begin; it < k_end; ++it) {
        mbar_wait(full_bar(st.stage), st.phase);
        float4* tile4 = reinterpret_cast<float4*>(gen_base + (size_t)st.stage * kStageBytes);
#pragma unroll 4
        for (int j = 0; j < kStageBytes / 16 / 128; ++j) {
          float4 v = tile4[ct + 128 * j];
          uint32_t r0, r1, r2, r3;
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r0) : "f"(v.x));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r1) : "f"(v.y));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r2) : "f"(v.z));
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r3) : "f"(v.w));
          tile4[ct + 128 * j] = make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float(r2), __uint_as_float(r3));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(conv_bar(st.stage));
        st.advance(S);
      }
    }
  } else {
    // TMEM lane quadrant q = accumulator rows 32q .. 32q+31 = mn-block q = tap row dy = q - 1; q = 3 is the unused shift
    const int q = warp & 3;
    int lt = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++lt) {
      int cc, n0, k_begin, k_end;
      decode_tile(tile, cc, n0, k_begin, k_end);
      const int acc = lt % kNAcc;
      const uint32_t acc_phase = (uint32_t)(lt / kNAcc) & 1u;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      if (q < 3) {
        const int c = cc * 32 + lane;
#pragma unroll 1
        for (int i = 0; i < 3; ++i) {
          const int t = q * 3 + i;
#pragma unroll 1
          for (int c0 = 0; c0 < BN; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * kAccCols + i * BN + c0), v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float* dst = a.gp + ((size_t)(n0 + c0 + j) * 9 + t) * Ctot + c;
              if (a.ksplit > 1) atomicAdd(dst, __uint_as_float(v[j]));
              else *dst = __uint_as_float(v[j]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

template <int BN>
int launch_wg_halo(const CUtensorMap& mX1, const CUtensorMap& mX2, const CUtensorMap& mDz, WgArgs& a, cudaStream_t st) {
  constexpr int stage_bytes = wgh_stage_bytes(BN);
  int stages = (210 * 1024) / stage_bytes;
  if (stages > 8) stages = 8;
  if (stages > a.kper) stages = a.kper < 2 ? 2 : a.kper;
  a.stages = stages;
  size_t smem = 1024 + (size_t)stages * stage_bytes + 8 * (3 * stages + 4) + 16;
  static bool attr_set = false;
  if (!attr_set) {
    MTD_CUDA(cudaFuncSetAttribute(wgrad_halo_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  int grid = a.n_tiles < mtd_sm_count() ? a.n_tiles : mtd_sm_count();
  mtd_launch(wgrad_halo_kernel<BN>, grid, kThreads, smem, st, mX1, mX2, mDz, a);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

__global__ void round_tf32_kernel(float* __restrict__ p, size_t n) {
  mtd_pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(p[i]));
    p[i] = __uint_as_float(r);
  }
}

}  // namespace

extern "C" {

// 1 = A operand through shared memory (conv_tc_kernel), 2 = A operand through TMEM with several pixel tiles per CTA
// (conv_tc2_kernel).  Process-wide; returns the previous value.
int mtd_tc_set_version(int version) {
  int prev = g_tc_version;
  if (version == 1 || version == 2) g_tc_version = version;
  return prev;
}

// Tuning hook (tools/tune_tc.py): force the Cout tile width and/or the stream-K piece length (k-steps per CTA; -1 =
// whole tiles only) of the forward/dgrad tensor-core kernel; 0 = let the cost model decide.
int mtd_tc_set_tuning(int bn, int sk_per) {
  if (bn != 0 && bn != 32 && bn != 64 && bn != 128) return MTD_EINVAL;
  g_tune_bn = bn; g_tune_per = sk_per;
  return MTD_OK;
}

// 1 (default): 3x3 / stride-1 layers with more than 32 channels run on the general halo-tile kernel (conv_halo_kernel);
// 0: on the tap-streaming kernel.
int mtd_tc_set_halo(int enabled) {
  const int prev = g_halo_enabled;
  g_halo_enabled = enabled ? 1 : 0;
  return prev;
}

// 1 (default): 32 -> 32 channel 3x3 layers run on the halo-tile kernel (conv_c32_kernel); 0: on the general kernel.
int mtd_tc_set_c32(int enabled) {
  const int prev = g_c32_enabled;
  g_c32_enabled = enabled ? 1 : 0;
  return prev;
}

int mtd_conv_fwd_tc_supported(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad) {
  int tw, th, tb;
  return tc_geometry(B, H, W, C1, C2, N, kh, kw, stride, pad, &tw, &th, &tb) && get_encode() != nullptr ? 1 : 0;
}

// Rounds a packed weight buffer to TF32 (round to nearest, ties away) in place — the B operand of the
// tensor-core kernels must be pre-rounded because tcgen05 truncates.
int mtd_round_tf32(float* p, long long n, void* stream) {
  MTD_REQUIRE(p && n > 0);
  int blocks = (int)(((size_t)n + 255) / 256);
  if (blocks > mtd_sm_count() * 16) blocks = mtd_sm_count() * 16;
  mtd_launch(round_tf32_kernel, blocks, 256, 0, (cudaStream_t)stream, p, (size_t)n);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

// In place: hi <- rna_tf32(w), lo <- rna_tf32(w - hi).  `lo` normally points n floats past `hi`.
int mtd_split_tf32(float* hi, float* lo, long long n, void* stream) {
  MTD_REQUIRE(hi && lo && n > 0);
  int blocks = (int)(((size_t)n + 255) / 256);
  if (blocks > mtd_sm_count() * 16) blocks = mtd_sm_count() * 16;
  mtd_launch(split_tf32_kernel, blocks, 256, 0, (cudaStream_t)stream, hi, lo, (size_t)n);
  MTD_CHECK_LAUNCH();
  return MTD_OK;
}

int mtd_conv_fwd_tc(const float* x1, const float* x2, const float* wp, const float* bias, const float* scale, int scale_group,
                    float* y,
                    float* aux, const float* add1, const float* add2, int B, int H, int W, int C1, int C2, int N, int kh,
                    int kw, int stride, int pad, int pre_act, int post_act, float slope, int passes, float* ws, long long ws_floats,
                    void* stream) {
  MTD_REQUIRE(x1 && wp && y && ((C2 == 0) == (x2 == nullptr)));
  int tw, th, tb;
  if (!tc_geometry(B, H, W, C1, C2, N, kh, kw, stride, pad, &tw, &th, &tb)) return MTD_EINVAL;
  TcArgs a{};
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  a.B = B; a.H = Ho; a.W = Wo; a.C1 = C1; a.C2 = C2; a.N = N; a.T = kh * kw;     // a.H / a.W: the output (tile) grid
  a.inH = H; a.inW = W; a.es = stride;
  for (int ky = 0; ky < kh; ++ky)
    for (int kx = 0; kx < kw; ++kx) { a.dy[ky * kw + kx] = ky - pad; a.dx[ky * kw + kx] = kx - pad; }
  a.out = y; a.scale = scale; a.scale_group = (scale && scale_group > 0 && scale_group < B) ? scale_group : 0;
  a.bias = bias; a.pre_act = pre_act; a.add1 = add1; a.add2 = add2; a.post_act = post_act;
  a.mask_src = nullptr; a.mask_act = 0; a.slope = slope; a.aux = aux;
  a.wrows_total = N;
  a.outH = Ho; a.outW = Wo; a.omy = a.omx = 1; a.ooy = a.oox = 0;
  a.ws = ws; a.ws_floats = ws ? ws_floats : 0;
  return launch_tc(x1, x2, wp, passes, a, (cudaStream_t)stream);
}

// Data gradient on the tensor cores: dx = (scale * dgrad(dz) + add1 + add2) * act'(mask_src).
// stride 1: dz (B,H,W,Cout), wpd[Cin][kh*kw][Cout].  stride 2 (4x4, pad 1): dz (B,H/2,W/2,Cout),
// wpd[4][Cin][4][Cout]: four output-parity classes, each a 2x2-tap stride-1 conv over dz scattered to
// (2i+py, 2j+px).  (H, W) are the conv INPUT dims = dx dims.
int mtd_conv_dgrad_tc(const float* dz, const float* wpd, float* dx, const float* scale, int scale_group, const float* add1,
                      const float* add2,
                      const float* mask_src, int mask_act, float slope, int B, int H, int W, int Cin, int Cout, int kh, int kw,
                      int stride, int pad, int passes, int cin_total, float* dx2, int c_split, float* ws, long long ws_floats,
                      void* stream) {
  MTD_REQUIRE(dz && wpd && dx);
  if (dx2) {      // two outputs: dx gets input channels [0, c_split), dx2 the rest (the two sources of a torch.cat layer)
    MTD_REQUIRE(g_tc_version == 1 && stride == 1 && c_split > 0 && c_split < Cin && c_split % 32 == 0 && (Cin - c_split) % 32 == 0 &&
                cin_total == Cin && !add1 && !add2 && !mask_src && mtd_aligned16(dx2));
  }
  cudaStream_t st = (cudaStream_t)stream;
  int tw, th, tb;
  TcArgs a{};
  a.ws = ws; a.ws_floats = ws ? ws_floats : 0;
  a.B = B; a.C1 = Cout; a.C2 = 0; a.N = Cin;
  a.out = dx; a.out2 = dx2; a.n_split = dx2 ? c_split : 0;
  a.scale = scale; a.scale_group = (scale && scale_group > 0 && scale_group < B) ? scale_group : 0;
  a.bias = nullptr; a.pre_act = 0; a.add1 = add1; a.add2 = add2; a.post_act = 0;
  a.mask_src = mask_src; a.mask_act = mask_act; a.slope = slope; a.aux = nullptr;
  a.outH = H; a.outW = W;
  if (stride == 1) {
    if (!tc_geometry(B, H, W, Cout, 0, Cin, kh, kw, 1, pad, &tw, &th, &tb)) return MTD_EINVAL;
    a.H = H; a.W = W; a.T = kh * kw;
    for (int ky = 0; ky < kh; ++ky)
      for (int kx = 0; kx < kw; ++kx) { a.dy[ky * kw + kx] = pad - ky; a.dx[ky * kw + kx] = pad - kx; }
    a.omy = a.omx = 1; a.ooy = a.oox = 0;
    a.wrows_total = cin_total;    // wpd may point at a row slice [cin_off, cin_off + Cin) of the [cin_total][T][Cout] pack
    return launch_tc(dz, nullptr, wpd, passes, a, st);
  }
  MTD_REQUIRE(stride == 2 && kh == 4 && kw == 4 && pad == 1 && H % 2 == 0 && W % 2 == 0 && cin_total == Cin);
  if (!tc_geometry(B, H / 2, W / 2, Cout, 0, Cin, 1, 1, 1, 0, &tw, &th, &tb)) return MTD_EINVAL;
  a.H = H / 2; a.W = W / 2; a.T = 4; a.omy = a.omx = 2;
  const size_t total = (size_t)B * H * W * Cin;
  const size_t cls_elems = (size_t)Cin * 4 * Cout;
  if (g_tc_version != 2) {
    // v1 kernel: the four output-parity classes are ONE launch (tile index carries the class); the classes own
    // disjoint output pixels, so whole tiles and stream-K pieces are finished exactly as for a stride-1 layer
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px)
        for (int aa = 0; aa < 2; ++aa)
          for (int bb = 0; bb < 2; ++bb) {
            const int ky = (1 - py) + 2 * aa, kx = (1 - px) + 2 * bb, i = (py * 2 + px) * 4 + aa * 2 + bb;
            a.dy[i] = (py + 1 - ky) / 2;
            a.dx[i] = (px + 1 - kx) / 2;
          }
    a.n_cls = 4;
    a.wrows_total = 4 * Cin;          // packed layout [4 classes][Cin][4][Cout]; the lo copy follows all four classes
    return launch_tc(dz, nullptr, wpd, passes, a, st);
  }
  int ksplit = 0;
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      TcArgs c = a;
      for (int aa = 0; aa < 2; ++aa)
        for (int bb = 0; bb < 2; ++bb) {
          int ky = (1 - py) + 2 * aa, kx = (1 - px) + 2 * bb;
          c.dy[aa * 2 + bb] = (py + 1 - ky) / 2;
          c.dx[aa * 2 + bb] = (px + 1 - kx) / 2;
        }
      c.ooy = py; c.oox = px;
      // packed layout [4 classes][Cin][4][Cout]; for passes == 3 the lo half starts after all four classes
      c.wrows_total = 4 * Cin;                            // rows from this class's base to the lo copy of the same class
      if (py == 0 && px == 0) {
        // decide the split once so all classes agree; zero dx up front when partial sums will be accumulated
        TcArgs probe = c;
        probe.n_wt = probe.W / tw; probe.n_ht = probe.H / th; probe.n_bt = (B + tb - 1) / tb;
        int m_tiles = probe.n_wt * probe.n_ht * probe.n_bt, kiters = 4 * (Cout / 32), bn_unused = 32;
        choose_tiling_v2(m_tiles, Cin, kiters, passes, 0, &bn_unused, &ksplit);
        if (ksplit > 1) MTD_CUDA(cudaMemsetAsync(dx, 0, total * sizeof(float), st));
      }
      int rc = launch_tc(dz, nullptr, wpd + (size_t)(py * 2 + px) * cls_elems, passes, c, st, ksplit, false);
      if (rc) return rc;
      if (c.ksplit != ksplit) return MTD_EINVAL;
    }
  if (ksplit > 1) {
    int blocks = (int)((total + 255) / 256);
    if (blocks > mtd_sm_count() * 8) blocks = mtd_sm_count() * 8;
    mtd_launch(tc_finish_kernel, blocks, 256, 0, st, a, total);
    MTD_CHECK_LAUNCH();
  }
  // ksplit == 1: the per-class epilogues already applied scale / adds / mask (each output pixel belongs to one class)
  return MTD_OK;
}

int mtd_conv_wgrad_tc_supported(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad) {
  int tw, th, tb;
  return wg_geometry(B, H, W, C1, C2, N, kh, kw, stride, pad, 64, &tw, &th, &tb) && get_encode() != nullptr ? 1 : 0;
}

// Plan of one weight-gradient call.  Kernel by shape: every 3x3 / stride-1 / pad-1 layer with an output grid of at
// least 8 x 8 in plain TF32 runs on the halo kernel, everything else on the tap-streaming kernel.  Run alone, the halo
// kernel is slower than the tap-streaming one at some Cout >= 128 shapes (profiles/r04_wgrad_new_{halo,taps}.txt), but
// in the train step the weight gradients run on a side stream beside the data gradients, and there its 2.3-3.2x lower
// L2 traffic and fewer CTAs win: the step is 0.35 ms faster with the halo kernel on every shape it runs than with a
// per-shape choice of the faster kernel in isolation (profiles/r04_bench_n1_select_*.json).
// Cout tile BN and split over pixels by a cost model (us):
//   T = 6 + waves * (2.5 + kper * ts) [+ 3 + 0.33 * ksplit * outputs / 64 K when split]
// A split adds a memset of the gradient and one fp32 atomic per output element per piece, so layers with few pixels
// and large weights (the deep discriminator layers) are not split.  ts = one k-step: on the tap-streaming kernel the
// L2 -> SM time of its stage at ~32 B/clk/SM; on the halo kernel the measured k-step (tools/bench_wgrad.py sweeps,
// profiles/r04_wgrad_sweep*.txt): 0.95 / 1.2 / 1.7 us at BN = 32 / 64 / 128, bound by its 24 MMAs and shared-memory
// traffic rather than by L2.  The tap-streaming kernel keeps its widest dz tile (x, its 9x re-read operand, is
// streamed once per n-tile).  MTD_WG_BN and MTD_WG_KSPLIT force the Cout tile and the split (tuning and test overrides).
static bool wg_plan(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad, int passes, WgArgs& out,
                    bool& out_halo, int& out_bn) {
  const int kp = passes == 3 ? 32 : 64;
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  const bool halo = passes == 1 && kh == 3 && kw == 3 && stride == 1 && pad == 1 && Ho >= kHaloPx && Wo >= kHaloPx;
  const int forced_bn = getenv("MTD_WG_BN") ? atoi(getenv("MTD_WG_BN")) : 0;
  const int forced_ks = getenv("MTD_WG_KSPLIT") ? atoi(getenv("MTD_WG_KSPLIT")) : 0;
  const int sms = mtd_sm_count();
  double best = 1e30;
  out_bn = 0;
  WgArgs a{};
  if (!wg_geometry(B, H, W, C1, C2, N, kh, kw, stride, pad, kp, &a.TW, &a.TH, &a.TB)) return false;
  if (halo) { a.TW = a.TH = kHaloPx; a.TB = 1; }
  a.B = B; a.H = Ho; a.W = Wo; a.C1 = C1; a.C2 = C2; a.N = N; a.T = kh * kw; a.es = stride;
  for (int ky = 0; ky < kh; ++ky)
    for (int kx = 0; kx < kw; ++kx) { a.dy[ky * kw + kx] = ky - pad; a.dx[ky * kw + kx] = kx - pad; }
  a.n_wt = Wo / a.TW; a.n_ht = Ho / a.TH; a.n_bt = (B + a.TB - 1) / a.TB;
  a.ptiles = a.n_wt * a.n_ht * a.n_bt;
  a.kc1 = C1 / 32; a.kc2 = C2 / 32;
  a.units = a.T * (a.kc1 + a.kc2);
  a.m_tiles = halo ? a.kc1 + a.kc2 : (a.units + 3) / 4;      // halo: one tile row = one 32-channel chunk, all 9 taps
  const int ks_max = a.ptiles / 2 > 1 ? a.ptiles / 2 : 1;
  for (int bn = 128; bn >= 32; bn /= 2) {
    if (N % bn) continue;
    if (forced_bn > 0 ? bn != forced_bn : !halo && bn != (N >= 128 ? 128 : N >= 64 ? 64 : 32)) continue;
    const int mn = a.m_tiles * (N / bn);
    const double ts = halo ? (bn == 128 ? 1.7 : bn == 64 ? 1.2 : 0.95)
                           : (128.0 + bn) * kp * 4.0 * (passes == 3 ? 2 : 1) / 61000.0;
    const double outputs = halo ? (double)a.units * 32.0 * N : (double)a.m_tiles * 128.0 * N;
    for (int ks0 = 1; ks0 <= ks_max && ks0 <= 512; ++ks0) {
      const int kper = (a.ptiles + ks0 - 1) / ks0;
      const int ks = (a.ptiles + kper - 1) / kper;
      if (forced_ks > 0 && kper != (a.ptiles + min(forced_ks, ks_max) - 1) / min(forced_ks, ks_max)) continue;
      const int waves = (mn * ks + sms - 1) / sms;
      double cost = 6.0 + waves * (2.5 + kper * ts);
      if (ks > 1) cost += 3.0 + 0.33 * ks * outputs / 65536.0;
      if (cost < best) {
        best = cost; out = a; out_halo = halo; out_bn = bn;
        out.ksplit = ks; out.kper = kper;
      }
    }
  }
  if (!out_bn) return false;
  out.n_nt = N / out_bn;
  out.n_tiles = out.m_tiles * out.n_nt * out.ksplit;
  return true;
}

// The plan mtd_conv_wgrad_tc runs for these arguments: plan[0] = 1 (halo kernel) / 0 (tap-streaming kernel),
// plan[1] = Cout tile BN, plan[2] = split over pixels, plan[3] = pixel tiles per piece, plan[4] = CTAs.
int mtd_conv_wgrad_tc_plan(int B, int H, int W, int C1, int C2, int N, int kh, int kw, int stride, int pad, int passes,
                           int* plan) {
  MTD_REQUIRE(plan && (passes == 1 || passes == 3));
  WgArgs a{};
  bool halo;
  int BN;
  if (!wg_plan(B, H, W, C1, C2, N, kh, kw, stride, pad, passes, a, halo, BN)) return MTD_EINVAL;
  plan[0] = halo ? 1 : 0; plan[1] = BN; plan[2] = a.ksplit; plan[3] = a.kper;
  plan[4] = a.n_tiles < mtd_sm_count() ? a.n_tiles : mtd_sm_count();
  return MTD_OK;
}

// gp[N][kh*kw][C1+C2] = sum over pixels of dz (x) x on the tensor cores (stride-1 "same" convs).
int mtd_conv_wgrad_tc(const float* x1, const float* x2, const float* dz, float* gp, int B, int H, int W, int C1, int C2, int N,
                      int kh, int kw, int stride, int pad, int passes, void* stream) {
  MTD_REQUIRE(x1 && dz && gp && ((C2 == 0) == (x2 == nullptr)) && (passes == 1 || passes == 3));
  cudaStream_t st = (cudaStream_t)stream;
  WgArgs a{};
  bool halo;
  int BN;
  if (!wg_plan(B, H, W, C1, C2, N, kh, kw, stride, pad, passes, a, halo, BN)) return MTD_EINVAL;
  if (!mtd_aligned16(x1) || !mtd_aligned16(dz) || (x2 && !mtd_aligned16(x2))) return MTD_EALIGN;
  a.gp = gp;
  if (a.ksplit > 1) MTD_CUDA(cudaMemsetAsync(gp, 0, (size_t)N * a.T * (C1 + C2) * sizeof(float), st));
  CUtensorMap mX1, mX2, mDz;
  const int xth = halo ? kHaloPx + 2 : a.TH;                   // halo: 10-row boxes starting one row above the tile
  int rc = make_act_map(&mX1, x1, C1, W, H, B, a.TW, xth, a.TB, true, stride);
  if (rc) return rc;
  if (C2) { rc = make_act_map(&mX2, x2, C2, W, H, B, a.TW, xth, a.TB, true, stride); if (rc) return rc; }
  else mX2 = mX1;
  rc = make_act_map(&mDz, dz, N, a.W, a.H, B, a.TW, a.TH, a.TB, true);
  if (rc) return rc;
  if (halo) {
    if (BN == 128) rc = launch_wg_halo<128>(mX1, mX2, mDz, a, st);
    else if (BN == 64) rc = launch_wg_halo<64>(mX1, mX2, mDz, a, st);
    else rc = launch_wg_halo<32>(mX1, mX2, mDz, a, st);
    return rc;
  }
#define WG_DISPATCH(BN_) rc = passes == 3 ? launch_wg<BN_, 3, 32>(mX1, mX2, mDz, a, st) : launch_wg<BN_, 1, 64>(mX1, mX2, mDz, a, st)
  if (BN == 128) { WG_DISPATCH(128); }
  else if (BN == 64) { WG_DISPATCH(64); }
  else { WG_DISPATCH(32); }
#undef WG_DISPATCH
  return rc;
}

}  // extern "C"
