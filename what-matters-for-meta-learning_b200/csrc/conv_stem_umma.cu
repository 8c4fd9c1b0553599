// The 5x5 stride-2 stem convolution of the 1-channel tasks (networks/ResNet.py conv1: 1 -> 64 channels,
// 128x128 -> 64x64) on tcgen05.  K = 25 taps is padded to ONE 32-wide K-block, so both kernels are a single
// K-block (forward) or a pixel contraction (weight gradient) around an im2col tile that the threads build
// from the NCHW image; what bounds them is the NHWC stream on the other side (forward: 1 MB written per
// image, weight gradient: 1 MB of dY read per image), not the 1600 FMAs per pixel the CUDA-core kernel
// (conv_small.cu, kept for fp32 mode and the 3-channel / 3x3 variants) spends.
//
//   forward  D[128 pixels x 64 co]  = Xcol[128 x 32] * W[64 x 32]^T           (K-major, SWIZZLE_128B)
//   wgrad    D[(hi|lo) co x 32 taps] += dY^T[co x 32 pixels] * Xcol[32 pixels x 32 taps]   (MN-major)
//
// 3xTF32 (see umma.cuh) is folded into the operand tiles instead of into extra instructions:
//   forward  B = [W_hi ; W_lo] stacked along N (128 rows): one N = 128 MMA gives X_hi*W_hi | X_hi*W_lo,
//            X_lo * W_hi (N = 64) is added to the cross-term columns.
//   wgrad    A = [dY_hi ; dY_lo] stacked along M, B = [Xcol_hi | Xcol_lo] stacked along N: ONE M=128, N=64
//            MMA per 8 pixels yields all four products; the epilogue adds the quadrants.  K index 25 of
//            Xcol is a constant 1, so column 25 of the result is the bias gradient.
#include <stdlib.h>

#include "common.cuh"
#include "umma.cuh"

namespace b200np {

using namespace umma;

namespace {

constexpr int kTaps = 25;

constexpr uint32_t tf32_idesc(int M, int N, bool mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (mn_major ? ((1u << 15) | (1u << 16)) : 0u) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// MN-major SWIZZLE_128B_BASE32B (see tapconv_umma.cu): 32-wide blocks LBO = 4096 B apart, 4-row groups
// SBO = 512 B apart, 32-byte swizzle units
__device__ __forceinline__ uint64_t mn_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(4096 >> 4) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(1) << 61;
  return d;
}
__device__ __forceinline__ uint32_t mn_off(int block, int k, int chunk) {
  return static_cast<uint32_t>(block * 4096 + (k >> 2) * 512 + (k & 3) * 128 + (((chunk >> 1) ^ (k & 3)) << 5) +
                               ((chunk & 1) << 4));
}
__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~uintptr_t(1023));
}

// ------------------------------------------------------------------------------------------------
// forward.  Persistent CTAs of 128 threads, four per SM (48 KB of shared memory, 128 TMEM columns
// each): a CTA is latency-bound (gather -> stage -> MMA -> epilogue), four of them interleave.
// thread = output pixel = row of the im2col tile = TMEM lane.
// ------------------------------------------------------------------------------------------------
template <bool X3>
__global__ void __launch_bounds__(128, 4)
    stem_fwd_umma_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                         float* __restrict__ y, uint32_t* __restrict__ relu_bits, int N, int H, int W, int relu,
                         long long tiles) {
  constexpr uint32_t kA = 128 * 32 * 4, kB = 64 * 32 * 4;
  constexpr uint32_t kCols = X3 ? 128 : 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* a_hi = smem;
  uint8_t* a_lo = smem + kA;
  uint8_t* b_hi = smem + 2 * kA;  // a_lo doubles as epilogue staging in single-pass mode
  uint8_t* b_lo = b_hi + kB;
  float* bias_s = reinterpret_cast<float*>(b_hi + 2 * kB);
  uint64_t* bar = reinterpret_cast<uint64_t*>(bias_s + 64);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform
  const uint32_t leader = elect_one_sync();
  const int OH = H / 2, OW = W / 2;
  const long long M = (long long)N * OH * OW;

  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  {  // weights [co][25] -> K-major rows of 32 (taps 25..31 zero), hi and lo planes; resident for the whole kernel
    const int co = tid >> 1, half = tid & 1;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k0 = (half * 4 + c) * 4;
      float4 v;
      v.x = k0 + 0 < kTaps ? __ldg(w + co * kTaps + k0 + 0) : 0.f;
      v.y = k0 + 1 < kTaps ? __ldg(w + co * kTaps + k0 + 1) : 0.f;
      v.z = k0 + 2 < kTaps ? __ldg(w + co * kTaps + k0 + 2) : 0.f;
      v.w = k0 + 3 < kTaps ? __ldg(w + co * kTaps + k0 + 3) : 0.f;
      split_store(b_hi, b_lo, sw128_offset(co, half * 4 + c), v, X3);
    }
    if (tid < 64) bias_s[tid] = __ldg(bias + tid);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  float v[28];
#pragma unroll
  for (int i = kTaps; i < 28; ++i) v[i] = 0.f;
  auto fetch = [&](long long tile) {
    const long long p = tile * 128 + tid;
    if (p < M) {
      const int ox = (int)(p % OW);
      const long long q = p / OW;
      const int oy = (int)(q % OH);
      const float* img = x + (q / OH) * H * W;
#pragma unroll
      for (int r = 0; r < 5; ++r) {
        const int iy = oy * 2 + r - 2;
        const bool rok = iy >= 0 && iy < H;
#pragma unroll
        for (int s = 0; s < 5; ++s) {
          const int ix = ox * 2 + s - 2;
          v[r * 5 + s] = (rok && ix >= 0 && ix < W) ? __ldg(img + (long long)iy * W + ix) : 0.f;
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < kTaps; ++i) v[i] = 0.f;
    }
  };

  long long tile = blockIdx.x;
  uint32_t phase = 0;
  if (tile < tiles) fetch(tile);
  for (; tile < tiles; tile += gridDim.x) {
#pragma unroll
    for (int c = 0; c < 7; ++c)
      split_store(a_hi, a_lo, sw128_offset(tid, c), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]), X3);
    split_store(a_hi, a_lo, sw128_offset(tid, 7), make_float4(0.f, 0.f, 0.f, 0.f), X3);
    fence_proxy_async();
    tc_fence_before();  // orders the previous tile's TMEM reads before this tile's MMAs
    __syncthreads();
    if (warp_u == 0) {  // all 32 lanes: descriptors stay in uniform registers, the elected lane issues
      tc_fence_after();
      const uint64_t ah = make_kmajor_sw128_desc(smem_u32(a_hi)), bh = make_kmajor_sw128_desc(smem_u32(b_hi));
      if (X3) {
        const uint64_t al = make_kmajor_sw128_desc(smem_u32(a_lo));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_tf32(tmem_d, ah + 2 * k, bh + 2 * k, tf32_idesc(128, 128, false), k != 0, leader);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_tf32(tmem_d + 64, al + 2 * k, bh + 2 * k, tf32_idesc(128, 64, false), 1u, leader);
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_tf32(tmem_d, ah + 2 * k, bh + 2 * k, tf32_idesc(128, 64, false), k != 0, leader);
      }
      umma_commit(bar, leader);
    }
    if (tile + gridDim.x < tiles) fetch(tile + gridDim.x);  // next tile's loads fly during the MMAs and the epilogue
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    // Epilogue.  A thread holds the 64 channels of ONE pixel; stored directly, a warp-wide 16-byte store
    // would touch 32 different 128-byte lines (half-written sectors, 32 L1 wavefronts).  The warp instead
    // transposes its 32 x 64 tile through the shared memory of its own im2col rows (idle until the next
    // tile is staged) and writes 512 contiguous bytes per instruction.
    const uint32_t taddr = tmem_d + (static_cast<uint32_t>(warp * 32) << 16);
    const int lane = tid & 31;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      uint32_t r[32];
      float acc[32];
      if (X3) {
        tmem_ld32(taddr + 64 + half * 32, r);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = __uint_as_float(r[j]);
        tmem_ld32(taddr + half * 32, r);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r[j]);
      } else {
        tmem_ld32(taddr + half * 32, r);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = __uint_as_float(r[j]);
      }
      uint8_t* piece = (half ? a_lo : a_hi) + warp * 4096 + lane * 128;
      uint32_t gates = 0u;   // (y > 0) of this thread's pixel, channels 32 half .. 32 half + 31
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b4 = *reinterpret_cast<const float4*>(bias_s + half * 32 + 4 * j);
        float4 o = make_float4(acc[4 * j] + b4.x, acc[4 * j + 1] + b4.y, acc[4 * j + 2] + b4.z, acc[4 * j + 3] + b4.w);
        if (relu) o = make_float4(fmaxf(o.x, 0.f), fmaxf(o.y, 0.f), fmaxf(o.z, 0.f), fmaxf(o.w, 0.f));
        *reinterpret_cast<float4*>(piece + ((j ^ (lane & 7)) << 4)) = o;
        gates |= (uint32_t)((o.x > 0.f) | ((o.y > 0.f) << 1) | ((o.z > 0.f) << 2) | ((o.w > 0.f) << 3)) << (4 * j);
      }
      // 1-bit ReLU gates for the data gradient that ends in this tensor: [pixel][2] words (thread = pixel here)
      if (relu_bits && tile * 128 + tid < M) relu_bits[(tile * 128 + tid) * 2 + half] = gates;
    }
    __syncwarp();
    {
      const long long p_base = tile * 128 + warp * 32;
      const int c = lane & 15, h = c >> 3, j = c & 7;
      const uint8_t* piece = (h ? a_lo : a_hi) + warp * 4096;
#pragma unroll
      for (int it = 0; it < 16; ++it) {
        const int rr = it * 2 + (lane >> 4);
        const float4 o = *reinterpret_cast<const float4*>(piece + rr * 128 + ((j ^ (rr & 7)) << 4));
        if (p_base + rr < M) *reinterpret_cast<float4*>(y + (p_base + rr) * 64 + c * 4) = o;
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(kCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// weight (and bias) gradient.  One CTA per chunk of pixels, K-blocks of 32 pixels, two stages.
//   A stage (16 KB): MN-major, four 32-channel blocks: dY_hi co 0-31 | dY_hi co 32-63 | dY_lo ... | dY_lo ...
//   B stage ( 8 KB): MN-major, two 32-tap blocks: Xcol_hi | Xcol_lo
// Xcol: thread = (pixel k = tid / 4, quarter q = tid % 4) gathers 8 taps of that pixel; dY: lanes walk
// consecutive 16-byte chunks, so every warp load is 512 contiguous bytes.
// part[(chunk * 2 + hi|lo)][co][32]: summed (with the other chunks) by the reducer into dw[co][25], db[co].
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kWA = 4 * 4096, kWB = 2 * 4096, kWStage = kWA + kWB;

template <bool X3>
__global__ void __launch_bounds__(128, 4)
    stem_wgrad_umma_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ part, int N,
                           int H, int W, long long pix_per_chunk) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kWStage);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform
  const uint32_t leader = elect_one_sync();
  const int OH = H / 2, OW = W / 2;
  const long long M = (long long)N * OH * OW;
  const long long p_begin = (long long)blockIdx.x * pix_per_chunk;
  long long p_end = p_begin + pix_per_chunk;
  if (p_end > M) p_end = M;
  const long long KB = p_begin < p_end ? (p_end - p_begin + 31) / 32 : 0;

  if (tid == 0) {
    for (int s = 0; s < 3; ++s) mbar_init(bars + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(128)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (!X3) {  // single pass: the lo halves of the stacked operands stay zero
    for (int i = tid; i < 2 * (int)kWStage / 16; i += 128) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  const int k = tid >> 2, q = tid & 3;
  // this thread's pixel of the current fetch, walked incrementally (+32 pixels per K-block)
  long long f_p = p_begin + k, f_n, f_pb = p_begin;
  int f_ox, f_oy;
  {
    f_ox = (int)(f_p % OW);
    const long long t = f_p / OW;
    f_oy = (int)(t % OH);
    f_n = t / OH;
  }
  float4 dv0[4], dv1[4];
  float xv0[8], xv1[8];
  auto fetch = [&](float4 (&dv)[4], float (&xv)[8]) {
    // dY: lanes walk consecutive 16-byte chunks (a warp instruction reads 512 contiguous bytes = 2 pixels)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long pd = f_pb + 8 * warp + 2 * j + (lane >> 4);
      dv[j] = pd < p_end ? ldg4(dy + pd * 64 + (lane & 15) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    f_pb += 32;
    if (f_p < p_end) {
      const float* img = x + f_n * H * W;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int tap = q * 8 + e;
        const int r = (tap * 13) >> 6, s = tap - 5 * r;  // tap / 5, tap % 5 for tap < 32
        const int iy = f_oy * 2 + r - 2, ix = f_ox * 2 + s - 2;
        float val = 0.f;
        if (tap < kTaps) {
          if (iy >= 0 && iy < H && ix >= 0 && ix < W) val = __ldg(img + (long long)iy * W + ix);
        } else if (tap == kTaps) {
          val = 1.f;  // bias-gradient column
        }
        xv[e] = val;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) xv[e] = 0.f;
    }
    f_p += 32;
    f_ox += 32;
    while (f_ox >= OW) {
      f_ox -= OW;
      if (++f_oy == OH) { f_oy = 0; ++f_n; }
    }
  };

  if (KB > 0) fetch(dv0, xv0);
  if (KB > 1) fetch(dv1, xv1);
  auto step = [&](long long kb, float4 (&dv)[4], float (&xv)[8]) {
    const int s = (int)(kb & 1);
    const long long use = kb >> 1;
    if (use >= 1) mbar_wait(bars + s, (uint32_t)((use - 1) & 1));
    uint8_t* a = smem + s * kWStage;
    uint8_t* b = a + kWA;
    // bank-conflict-free 16-byte stores: the eight threads of a quarter-warp must hit eight different
    // 16-byte slots of the 128-byte line.  dY: a quarter-warp holds the eight chunks of one 32-channel block
    // of one pixel.  Xcol: odd pixels swap the two chunks.
#pragma unroll
    for (int j = 0; j < 4; ++j)
      split_store(a, a + 2 * 4096, mn_off((lane >> 3) & 1, 8 * warp + 2 * j + (lane >> 4), lane & 7), dv[j], X3);
    {
      const int sw = k & 1;
      const float4 c0 = make_float4(xv[0], xv[1], xv[2], xv[3]), c1 = make_float4(xv[4], xv[5], xv[6], xv[7]);
      split_store(b, b + 4096, mn_off(0, k, q * 2 + sw), sw ? c1 : c0, X3);
      split_store(b, b + 4096, mn_off(0, k, q * 2 + (sw ^ 1)), sw ? c0 : c1, X3);
    }
    fence_proxy_async();
    __syncthreads();
    if (warp_u == 0) {  // all 32 lanes: descriptors stay in uniform registers, the elected lane issues
      tc_fence_after();
      const uint64_t ad = mn_desc(smem_u32(a)), bd = mn_desc(smem_u32(b));
      const uint32_t d_blk = tmem_d + (uint32_t)(kb & 1) * 64;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)  // next 8 pixels: +1024 B
        umma_tf32(d_blk, ad + 64 * ks, bd + 64 * ks, tf32_idesc(128, X3 ? 64 : 32, true), (kb >= 2) | (ks != 0), leader);
      umma_commit(bars + s, leader);
      if (kb == KB - 1) umma_commit(bars + 2, leader);
    }
    if (kb + 2 < KB) fetch(dv, xv);
  };
  for (long long kb = 0; kb < KB; kb += 2) {
    step(kb, dv0, xv0);
    if (kb + 1 < KB) step(kb + 1, dv1, xv1);
  }

  // epilogue: lane = row m = (hi|lo) * 64 + co; add the two rotating blocks and the hi|lo tap columns
  if (KB > 0) {
    mbar_wait(bars + 2, 0);
    tc_fence_after();
  }
  {
    const uint32_t taddr = tmem_d + (static_cast<uint32_t>(warp * 32) << 16);
    float acc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) acc[j] = 0.f;
    uint32_t r[32];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int blk = i & 1, cross = i < 2;
      if (blk < KB && (X3 || !cross)) {
        tmem_ld32(taddr + blk * 64 + cross * 32, r);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r[j]);
      }
    }
    float* po = part + ((long long)blockIdx.x * 128 + tid) * 32;  // [chunk][hi|lo][co][32]
#pragma unroll
    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(po + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(128) : "memory");
  }
}

int stem_wgrad_chunks(long long M) {
  // CTAs per SM over the whole launch (4 are resident at a time); every CTA leaves a 16 KB partial for the reducer
  constexpr int per_sm = 4;   // one resident wave; 8: +38 us per step in reducer traffic, 2: tail
  long long want = (long long)per_sm * kNumSMs, maxc = ceil_div(M, 64);
  if (want > maxc) want = maxc;
  return (int)(want < 1 ? 1 : want);
}

template <typename K>
bool set_smem(K kernel, size_t smem) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
}

}  // namespace

bool stem_umma_supported(int Cin, int R, int Cout, int precision) {
  return precision != B200NP_PREC_FP32_SIMT && Cin == 1 && R == 5 && Cout == 64;
}

int launch_stem_fwd_umma(const float* x, const float* w, const float* bias, float* y, uint32_t* relu_bits, int N, int H,
                         int W, int relu, int precision, cudaStream_t st) {
  const bool x3 = precision != B200NP_PREC_TF32;
  const long long M = (long long)N * (H / 2) * (W / 2);
  const long long tiles = ceil_div(M, 128);
  const size_t smem = 2 * (128 * 32 * 4 + 64 * 32 * 4) + 256 + 64 + 1024;
  static bool configured = false;
  if (!configured) {
    if (!set_smem(stem_fwd_umma_kernel<true>, smem) || !set_smem(stem_fwd_umma_kernel<false>, smem))
      return B200NP_E_LAUNCH;
    configured = true;
  }
  const long long cap = 4LL * kNumSMs;
  const int grid = (int)(tiles < cap ? tiles : cap);
  if (x3) stem_fwd_umma_kernel<true><<<grid, 128, smem, st>>>(x, w, bias, y, relu_bits, N, H, W, relu, tiles);
  else stem_fwd_umma_kernel<false><<<grid, 128, smem, st>>>(x, w, bias, y, relu_bits, N, H, W, relu, tiles);
  return launch_status();
}

size_t stem_wgrad_umma_workspace(int N, int H, int W) {
  const long long M = (long long)N * (H / 2) * (W / 2);
  return (size_t)stem_wgrad_chunks(M) * 2 * 64 * 32 * sizeof(float);
}

int launch_stem_wgrad_umma(const float* x, const float* dy, float* dw, float* db, int N, int H, int W, int precision,
                           void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool x3 = precision != B200NP_PREC_TF32;
  const long long M = (long long)N * (H / 2) * (W / 2);
  const int chunks = stem_wgrad_chunks(M);
  if (!ws || ws_bytes < (size_t)chunks * 2 * 64 * 32 * sizeof(float)) return B200NP_E_WORKSPACE;
  const long long ppc = ceil_div(ceil_div(M, chunks), 32) * 32;
  const size_t smem = 2 * kWStage + 64 + 1024;
  static bool configured = false;
  if (!configured) {
    if (!set_smem(stem_wgrad_umma_kernel<true>, smem) || !set_smem(stem_wgrad_umma_kernel<false>, smem)) return B200NP_E_LAUNCH;
    configured = true;
  }
  if (x3) stem_wgrad_umma_kernel<true><<<chunks, 128, smem, st>>>(x, dy, (float*)ws, N, H, W, ppc);
  else stem_wgrad_umma_kernel<false><<<chunks, 128, smem, st>>>(x, dy, (float*)ws, N, H, W, ppc);
  int rc = launch_status();
  if (rc != B200NP_OK) return rc;
  return launch_reduce_partials((const float*)ws, dw, chunks * 2, 64 * 32, ReduceMap{2, kTaps, 32, 0, db}, st);
}

}  // namespace b200np
