// Weight gradient of a 3x3 stride-1 64->64 convolution (+ the fused 1x1 stride-2 skip projection) as a HALO kernel.
//
// The gather kernel (tapconv_umma.cu: tapwgrad_umma_kernel) stages x once per TAP and dY once per tap PAIR, and ncu
// shows the L1 data pipe -- global loads, shared-memory stores and the tensor core's operand reads share it -- 95 %
// busy at 32 % tensor activity (DESIGN.md, finding 12).  Here a CTA stages the x halo and the dY tile of a 4 x 16
// pixel tile ONCE and forms all its taps from them:
//   * planes [halo row][channel block][pixel][32 ch]: 128 B per pixel and block, hi and lo copies, stored with the
//     32-byte-unit swizzle of SWIZZLE_128B_BASE32B taken from absolute shared-memory address bits;
//   * a tap is a descriptor whose start is shifted by whole pixels, legal for MN-major operands from any 128-byte row
//     and with any 128-byte-multiple LBO (profiles/umma_mn_descriptor_probe_r1.txt);
//   * two taps are the halves of M = 128: the channel-block stride (LBO) is one block of one row, so the rows that
//     follow at 2 LBO supply the second tap;
//   * dY is [row][hi | lo][channel block][pixel]: one N = 128 MMA gives x_hi*dY_hi and x_hi*dY_lo, an N = 64 MMA adds
//     x_lo*dY_hi (the 3xTF32 scheme of the other kernels; single-pass tf32 uses one N = 64 MMA).
// Two CTA roles share a pixel chunk (TMEM holds the accumulators of three tap pairs, not of ten taps):
//   role 0: taps dy in {-1, 0}: halo rows r and r + 1 of one compact x halo are the two halves            (6 taps)
//   role 1: taps dy = +1, and the skip tap as the second half of the dx = 0 pair: rows are interleaved
//           [x row r + 1 | skip row r]; the second halves of the dx = -1 / +1 pairs are not used            (4 taps)
// Accumulators live in TMEM across all tiles of the chunk; partial tiles go to part[chunk][tap][co][ci] like the gather
// kernel's, so the same reduction follows.  Role 0 also sums dY for the bias gradient.
// Measured as a prototype (tools/probe/wgrad_halo_proto.cu, 12 tap-products): 0.69 ms against 0.80 ms for the 9 taps +
// reduction of the gather kernel at 1140 images.
//
// Warp-specialised CTA; full/empty mbarriers hand two stages over, so the tensor core works on tile i while the loader
// and the split warps prepare tile i+1:
//   warp 8      loader: per tile one cp.async.bulk.tensor per (row, 32-channel block) of the x halo, the skip rows and
//               the dY tile drops the raw fp32 pixels into the `hi` regions of a stage (4-D maps [channel][x][y][image],
//               box 32 x pixels x 1 x 1, SWIZZLE_128B_ATOM_32B = the MN-major operand swizzle; image borders arrive as
//               zeros) -- no global load, no address arithmetic in any thread;
//   warps 0-7   split warps, shared memory -> shared memory (split_sweep): the tf32 hi / lo operands and the dY column
//               sums for the bias gradient;
//   warp 9      MMA issuer only.  (A block-synchronous form, in which warp 0 issued a tile's 48 MMAs and then helped
//               stage the next one, paid T_tile = T_issue + T_store: 0.79 ms against 0.56 ms.)

#include "tapconv.cuh"
#include "tma.cuh"
#include "umma.cuh"

namespace b200np {

using namespace umma;

namespace {

constexpr int RT = 4, TW = 16, HW = TW + 2;
constexpr uint32_t S_A = HW * 128;                       // one channel block of one (halo) row: 2304 B
constexpr uint32_t A0_PLANE = (RT + 1) * 2 * S_A;        // role 0: hi (or lo) copy of the x halo, rows hr = 0..RT
constexpr uint32_t A1_PLANE = RT * 4 * S_A;              // role 1: [row][x cb0 | x cb1 | skip cb0 | skip cb1]
constexpr uint32_t S_B = TW * 128;                       // one channel block of one dY row: 2048 B
constexpr uint32_t B_TILE = RT * 4 * S_B;                // [row][hi | lo][block][pixel]
constexpr uint32_t STAGE = 2 * A1_PLANE + B_TILE;        // sized for role 1 (the larger): 106496 B = 104 * 1024
constexpr uint32_t kIdesc128x64 = kIdescTf32_128x64 | (1u << 15) | (1u << 16);
constexpr uint32_t kIdesc128x128 =
    (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
static_assert(A0_PLANE % 512 == 0 && A1_PLANE % 512 == 0 && STAGE % 1024 == 0, "swizzle phase of the regions");

struct HaloWgradArgs {
  const float* x;      // [N, H, W, 64]
  const float* dy;     // [N, H, W, 64]
  const float* xs;     // nullable: skip source [N, 2H, 2W, 64], read at (2 oy, 2 ox)
  float* part;         // [chunks][ntaps][co][ci]
  float* part_db;      // nullable: [chunks][64]
  int N, H, W, ntaps;  // ntaps = 9 or 10 (with skip)
  long long tiles, per;
};

__device__ __forceinline__ uint64_t mn_desc(uint32_t saddr, uint32_t lbo) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(lbo >> 4) << 16;   // next 32-channel block
  d |= static_cast<uint64_t>(512 >> 4) << 32;   // SBO: next group of 4 pixels
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(1) << 61;          // SWIZZLE_128B_BASE32B, base_offset 0
  return d;
}

struct HaloWgradTma {
  tma::Map x;     // [64][W][H][N]  box 32 x 18 x 1 x 1
  tma::Map dy;    // [64][W][H][N]  box 32 x 16 x 1 x 1
  tma::Map xs;    // parity-(0,0) view of the skip source [64][W][H][N] (strides doubled), box 32 x 16 x 1 x 1
};
constexpr int kSplitThreads = 256, kLoadWarp = 8, kIssueWarp = 9, kThreads = 320;

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ void mbar_arrive_(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// Split warps of the TMA-fed kernels: linear sweeps over the landed raw fp32 regions, one LDS + one STS per 16 bytes.
// fp32-grade mode: the raw region is the `hi` operand as it is (the tensor core truncates fp32 to tf32) and only
// lo = x - trunc_tf32(x) is written; single-pass mode rounds to nearest in place.  A: `a_units` 16-byte units whose lo
// copy sits A_PLANE bytes further; B: per row [hi cb0 | hi cb1 | lo cb0 | lo cb1] blocks of S_B bytes.
// Thread `tid` (< 256) of the B sweep always sees the same 16-byte position of a 128-byte row and the same swizzle
// phase, hence the same four channels: `dbs` accumulates their dY sums (bias gradient) when DB is set.
template <bool X3, bool DB>
__device__ __forceinline__ void split_sweep(uint32_t a_hi, uint32_t a_plane, uint32_t a_units, uint32_t b, int rows,
                                            int tid, float4& dbs) {
  for (uint32_t u0 = tid; u0 < a_units; u0 += 4 * kSplitThreads) {
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t u = u0 + j * kSplitThreads;
      if (u < a_units) v[j] = lds128(a_hi + u * 16u);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t u = u0 + j * kSplitThreads;
      if (u < a_units) {
        if (X3) sts128(a_hi + a_plane + u * 16u, lo_of_truncated(v[j]));
        else sts128(a_hi + u * 16u, to_tf32_4(v[j]));
      }
    }
  }
  // B: unit u = r * 256 + w, w < 256 = the two hi blocks of row r (2 * S_B / 16 units)
  static_assert(2 * S_B / 16 == kSplitThreads, "one B row per sweep pass");
  float4 y[4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
    if (r < rows) y[r] = lds128(b + (uint32_t)r * 4u * S_B + (uint32_t)tid * 16u);
#pragma unroll
  for (int r = 0; r < 4; ++r)
    if (r < rows) {
      const uint32_t addr = b + (uint32_t)r * 4u * S_B + (uint32_t)tid * 16u;
      if (X3) sts128(addr + 2u * S_B, lo_of_truncated(y[r]));
      else sts128(addr, to_tf32_4(y[r]));
      if (DB) { dbs.x += y[r].x; dbs.y += y[r].y; dbs.z += y[r].z; dbs.w += y[r].w; }
    }
}
// channel quadruple and reduction slot of thread `tid` in split_sweep's B pass (see there)
__device__ __forceinline__ void db_slot(int tid, int& channel, int& slot) {
  const int p = tid & 7, phase = (tid >> 3) & 3, cb = tid >> 7;
  const int chunk = (((p >> 1) ^ phase) << 1) | (p & 1);
  channel = cb * 32 + chunk * 4;
  slot = ((tid >> 5) & 3) * 4 + phase;
}

template <bool X3, int ROLE>
__device__ __forceinline__ void run_role_tma(const HaloWgradArgs& a, const HaloWgradTma& tm, uint8_t* smem, uint64_t* bars,
                                             uint32_t tmem) {
  constexpr uint32_t A_PLANE = ROLE == 0 ? A0_PLANE : A1_PLANE;
  constexpr uint32_t ROW_A = ROLE == 0 ? 2 * S_A : 4 * S_A;
  uint64_t* t_full = bars;        // [2] tensor copies landed              (count 1 + tx)
  uint64_t* s_full = bars + 2;    // [2] split warps done                  (count 256)
  uint64_t* s_empty = bars + 4;   // [2] the MMAs that read the stage retired (tcgen05.commit)
  uint64_t* done = bars + 6;      // all MMAs of the chunk retired
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int chunk = blockIdx.x;        // roles are blockIdx.y: two successive waves (0.28 + 0.29 ms alone).  Interleaving
                                       // the roles as neighbouring CTAs, so that the second reader of a chunk hits L2,
                                       // was measured at 0.58 -> 0.92 ms and reverted.
  const int H = a.H, W = a.W;
  const int tiles_x = W / TW, tiles_img = tiles_x * (H / RT);
  const long long t_begin = chunk * a.per, t_end = t_begin + a.per < a.tiles ? t_begin + a.per : a.tiles;
  float4 dbs = make_float4(0.f, 0.f, 0.f, 0.f);

  if (ROLE == 1) {
    // columns 0 and 17 of the skip blocks are never written; the unused second halves of the dx = -1 / +1 pairs read
    // them, so they must not hold NaN / Inf garbage: zero both stages once (before any tensor copy is issued)
    for (uint32_t o = tid * 16; o < 2 * STAGE; o += kThreads * 16) *reinterpret_cast<float4*>(smem + o) = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_proxy_async();
    __syncthreads();
  }

  if (warp == kLoadWarp) {
    // ===================== loader =====================
    const uint32_t leader = elect_one_sync();
    const bool skip = ROLE == 1 && a.xs != nullptr;
    const uint32_t kTx = ROLE == 0 ? ((RT + 1) * 2 * HW + RT * 2 * TW) * 128u
                                   : (RT * 2 * HW + RT * 2 * TW + (skip ? RT * 2 * TW : 0)) * 128u;
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it & 1);
      const int n = (int)(tile / tiles_img), rem = (int)(tile - (long long)n * tiles_img);
      const int oy0 = (rem / tiles_x) * RT, ox0 = (rem % tiles_x) * TW;
      if (it >= 2) mbar_wait(s_empty + s, (uint32_t)(((it >> 1) - 1) & 1));
      if (leader) mbar_expect_tx_(t_full + s, kTx);
      const uint32_t st = smem_u32(smem + s * STAGE), bar = smem_u32(t_full + s);
      const uint32_t b0 = st + 2 * A_PLANE;
      if (ROLE == 0) {
#pragma unroll
        for (int hr = 0; hr <= RT; ++hr)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb)
            tma::load_4d(st + (uint32_t)(hr * 2 + cb) * S_A, &tm.x, bar, cb * 32, ox0 - 1, oy0 + hr - 1, n, leader);
      } else {
#pragma unroll
        for (int r = 0; r < RT; ++r)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb) {
            tma::load_4d(st + (uint32_t)(r * 4 + cb) * S_A, &tm.x, bar, cb * 32, ox0 - 1, oy0 + r + 1, n, leader);
            // skip pixel k sits at column k + 1 of its block (the dx = 0 pair, start column 1, reads it)
            tma::load_4d(st + (uint32_t)(r * 4 + 2 + cb) * S_A + 128u, &tm.xs, bar, cb * 32, ox0, oy0 + r, n, skip ? leader : 0u);
          }
      }
#pragma unroll
      for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int cb = 0; cb < 2; ++cb)
          tma::load_4d(b0 + (uint32_t)(r * 4 + cb) * S_B, &tm.dy, bar, cb * 32, ox0, oy0 + r, n, leader);
    }
  } else if (warp == kIssueWarp) {
    // ===================== MMA issuer =====================
    const uint32_t leader = elect_one_sync();
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it & 1);
      const uint32_t par = (uint32_t)((it >> 1) & 1);
      mbar_wait(t_full + s, par);
      mbar_wait(s_full + s, par);
      tc_fence_after();
      const uint32_t a_hi = smem_u32(smem + s * STAGE), a_lo = a_hi + A_PLANE, b0 = a_hi + 2 * A_PLANE;
#pragma unroll
      for (int r = 0; r < RT; ++r) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const uint64_t bd = mn_desc(b0 + r * 4 * S_B + hf * 8 * 128, S_B);
#pragma unroll
          for (int j = 0; j < 3; ++j) {   // dx = j - 1: the (halo) column of output pixel k is hf*8 + k + j
            const uint32_t aoff = r * ROW_A + (hf * 8 + j) * 128;
            const uint32_t d = tmem + j * 128;
            const uint32_t acc = (it == 0 && r == 0 && hf == 0) ? 0u : 1u;
            if (X3) {
              umma_tf32(d, mn_desc(a_hi + aoff, S_A), bd, kIdesc128x128, acc, leader);
              umma_tf32(d + 64, mn_desc(a_lo + aoff, S_A), bd, kIdesc128x64, 1u, leader);
            } else {
              umma_tf32(d, mn_desc(a_hi + aoff, S_A), bd, kIdesc128x64, acc, leader);
            }
          }
        }
      }
      umma_commit(s_empty + s, leader);
      if (tile + 1 == t_end) umma_commit(done, leader);
    }
  } else {
    // ===================== split warps: smem -> smem =====================
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it & 1);
      mbar_wait(t_full + s, (uint32_t)((it >> 1) & 1));
      const uint32_t a_hi = smem_u32(smem + s * STAGE);
      split_sweep<X3, ROLE == 0>(a_hi, A_PLANE, A_PLANE / 16, a_hi + 2 * A_PLANE, RT, tid, dbs);
      fence_proxy_async();
      mbar_arrive_(s_full + s);
    }
  }
  // every chunk has at least one tile (the host sizes `per` that way)
  mbar_wait(done, 0);
  tc_fence_after();
  __syncthreads();
  if (ROLE == 0 && a.part_db) {   // all MMAs have retired: the stages are free for the 16-row reduction of the dY sums
    float* red = reinterpret_cast<float*>(smem);
    if (tid < kSplitThreads) {
      int channel, slot;
      db_slot(tid, channel, slot);
      *reinterpret_cast<float4*>(red + slot * 64 + channel) = dbs;
    }
    __syncthreads();
    if (tid < 64) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) t += red[r * 64 + tid];
      a.part_db[(long long)chunk * 64 + tid] = t;
    }
  }
  if (warp >= 8) return;
  // rows m = 32 q + lane = half_tap * 64 + ci; warps w and w + 4 share lane quarter q = w % 4 and take 32 co each
  const int q = warp & 3, half = warp >> 2, second = q >> 1, ci = (q & 1) * 32 + lane;
#pragma unroll 1
  for (int j = 0; j < 3; ++j) {
    int tap;
    if (ROLE == 0) tap = second * 3 + j;                                // (dy = -1 | 0, dx = j - 1)
    else tap = second ? ((j == 1 && a.ntaps > 9) ? 9 : -1) : 6 + j;     // (dy = +1, dx = j - 1) | the skip tap
    uint32_t r0[32], r1[32];
    const uint32_t ta = tmem + (static_cast<uint32_t>(q * 32) << 16) + j * 128 + half * 32;
    tmem_ld32(ta, r0);
    if (X3) tmem_ld32(ta + 64, r1);
    if (tap >= 0) {
      float* po = a.part + ((long long)chunk * a.ntaps + tap) * 64 * 64 + ci;
#pragma unroll
      for (int i = 0; i < 32; ++i)
        po[(half * 32 + i) * 64] = (X3 ? __uint_as_float(r1[i]) : 0.f) + __uint_as_float(r0[i]);
    }
  }
}

template <bool X3>
__global__ void __launch_bounds__(kThreads, 1) tapwgrad_halo_tma_kernel(const HaloWgradArgs a,
                                                                         const __grid_constant__ HaloWgradTma tm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * STAGE);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(bars + s, 1); mbar_init(bars + 2 + s, kSplitThreads); mbar_init(bars + 4 + s, 1); }
    mbar_init(bars + 6, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (blockIdx.y == 0) run_role_tma<X3, 0>(a, tm, smem, bars, tmem);
  else run_role_tma<X3, 1>(a, tm, smem, bars, tmem);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// ------------------------------------------------------------------------------------------------------------
// Stride-2 3x3 weight gradient (conv1 of a BasicBlock: x [N, 2H, 2W, 64], dY [N, H, W, 64]) in the same TMA-fed form.
// Tap (dy, dx) reads x[2 oy + dy][2 ox + dx] = parity plane (dy & 1, dx & 1) at shift ((dy - (dy & 1)) / 2, ...): the
// four parity views of x are four tensor maps (base shifted, strides doubled), each plane a dense stride-1 stencil source.
//   role 0: the vertical pairs (dy = -1 | dy = +1) for dx = -1, 0, +1: consecutive rows of the ODD-row planes are the two
//           halves of M = 128 (region Q: plane (1,1), 18 pixel slots per row, dx = -1 / +1 are starts 0 / 1; region P:
//           plane (1,0), dx = 0)                                                                           (6 taps)
//   role 1: dy = 0: (0,-1) | (0,+1) are one pair -- the even-row plane (0,1) is loaded twice, the second copy one pixel
//           further right, so one descriptor start serves both halves; (0,0) is a single whose second half is not used
//                                                                                                          (3 taps)
// Tiles are 2 x 16 output pixels (three x rows per tile and role fit three stages of 67 KB).
// ------------------------------------------------------------------------------------------------------------
namespace s2 {
constexpr int RT2 = 2, NST = 3;
constexpr uint32_t Q_BYTES = (RT2 + 1) * 2 * S_A;        // 13824
constexpr uint32_t P_BYTES = (RT2 + 1) * 2 * S_B;        // 12288
constexpr uint32_t E_BYTES = RT2 * 4 * S_B;              // 16384: [row][copy][block][pixel]
constexpr uint32_t Z_BYTES = RT2 * 2 * S_B;              //  8192
constexpr uint32_t A_PLANE = Q_BYTES + P_BYTES;          // 26112 >= E_BYTES + Z_BYTES (24576)
constexpr uint32_t B_TILE2 = RT2 * 4 * S_B;              // 16384
constexpr uint32_t STAGE2 = 2 * A_PLANE + B_TILE2;       // 68608
static_assert(Q_BYTES % 512 == 0 && A_PLANE % 512 == 0 && E_BYTES % 512 == 0 && STAGE2 % 1024 == 0 && E_BYTES + Z_BYTES <= A_PLANE, "layout");
}  // namespace s2

struct HaloWgradS2Tma {
  tma::Map x[4];  // parity views (py * 2 + px) of x: [64][W][H][N], box 32 x 18 (px = 1) | 16 (px = 0) x 1 x 1
  tma::Map dy;    // [64][W][H][N], box 32 x 16 x 1 x 1
};

template <bool X3, int ROLE>
__device__ __forceinline__ void run_role_s2(const HaloWgradArgs& a, const HaloWgradS2Tma& tm, uint8_t* smem, uint64_t* bars,
                                            uint32_t tmem) {
  using namespace s2;
  constexpr int NPAIR = ROLE == 0 ? 3 : 2;
  uint64_t* t_full = bars;             // [NST]
  uint64_t* s_full = bars + NST;       // [NST]
  uint64_t* s_empty = bars + 2 * NST;  // [NST]
  uint64_t* done = bars + 3 * NST;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int chunk = blockIdx.x;        // roles are blockIdx.y (see run_role_tma)
  const int H = a.H, W = a.W;          // dY geometry
  const int tiles_x = W / TW, tiles_img = tiles_x * (H / RT2);
  const long long t_begin = chunk * a.per, t_end = t_begin + a.per < a.tiles ? t_begin + a.per : a.tiles;
  float4 dbs = make_float4(0.f, 0.f, 0.f, 0.f);

  if (ROLE == 1) {   // the unused second half of the (0,0) single reads beyond region Z: keep it finite
    for (uint32_t o = tid * 16; o < NST * STAGE2; o += kThreads * 16) *reinterpret_cast<float4*>(smem + o) = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_proxy_async();
    __syncthreads();
  }

  if (warp == kLoadWarp) {
    const uint32_t leader = elect_one_sync();
    constexpr uint32_t kTx = ROLE == 0 ? ((RT2 + 1) * 2 * (HW + TW) + RT2 * 2 * TW) * 128u : (RT2 * 6 * TW + RT2 * 2 * TW) * 128u;
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it % NST);
      const int n = (int)(tile / tiles_img), rem = (int)(tile - (long long)n * tiles_img);
      const int oy0 = (rem / tiles_x) * RT2, ox0 = (rem % tiles_x) * TW;
      if (it >= NST) mbar_wait(s_empty + s, (uint32_t)((it / NST - 1) & 1));
      if (leader) mbar_expect_tx_(t_full + s, kTx);
      const uint32_t st = smem_u32(smem + s * STAGE2), bar = smem_u32(t_full + s);
      const uint32_t b0 = st + 2 * A_PLANE;
      if (ROLE == 0) {
#pragma unroll
        for (int hr = 0; hr <= RT2; ++hr)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb) {
            tma::load_4d(st + (uint32_t)(hr * 2 + cb) * S_A, &tm.x[3], bar, cb * 32, ox0 - 1, oy0 - 1 + hr, n, leader);
            tma::load_4d(st + Q_BYTES + (uint32_t)(hr * 2 + cb) * S_B, &tm.x[2], bar, cb * 32, ox0, oy0 - 1 + hr, n, leader);
          }
      } else {
#pragma unroll
        for (int r = 0; r < RT2; ++r)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb) {
            tma::load_4d(st + (uint32_t)(r * 4 + cb) * S_B, &tm.x[1], bar, cb * 32, ox0 - 1, oy0 + r, n, leader);       // dx = -1
            tma::load_4d(st + (uint32_t)(r * 4 + 2 + cb) * S_B, &tm.x[1], bar, cb * 32, ox0, oy0 + r, n, leader);       // dx = +1
            tma::load_4d(st + E_BYTES + (uint32_t)(r * 2 + cb) * S_B, &tm.x[0], bar, cb * 32, ox0, oy0 + r, n, leader); // (0, 0)
          }
      }
#pragma unroll
      for (int r = 0; r < RT2; ++r)
#pragma unroll
        for (int cb = 0; cb < 2; ++cb)
          tma::load_4d(b0 + (uint32_t)(r * 4 + cb) * S_B, &tm.dy, bar, cb * 32, ox0, oy0 + r, n, leader);
    }
  } else if (warp == kIssueWarp) {
    const uint32_t leader = elect_one_sync();
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it % NST);
      const uint32_t par = (uint32_t)((it / NST) & 1);
      mbar_wait(t_full + s, par);
      mbar_wait(s_full + s, par);
      tc_fence_after();
      const uint32_t a_hi = smem_u32(smem + s * STAGE2), a_lo = a_hi + A_PLANE, b0 = a_hi + 2 * A_PLANE;
#pragma unroll
      for (int r = 0; r < RT2; ++r) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const uint64_t bd = mn_desc(b0 + r * 4 * S_B + hf * 8 * 128, S_B);
#pragma unroll
          for (int j = 0; j < NPAIR; ++j) {
            uint32_t aoff, lbo;
            if (ROLE == 0) {
              if (j == 1) { aoff = Q_BYTES + r * 2 * S_B + hf * 8 * 128; lbo = S_B; }              // dx = 0: plane (1,0)
              else { aoff = r * 2 * S_A + (hf * 8 + (j == 2 ? 1 : 0)) * 128; lbo = S_A; }          // dx = -1 | +1: plane (1,1)
            } else {
              if (j == 0) { aoff = r * 4 * S_B + hf * 8 * 128; lbo = S_B; }                        // (0,-1) | (0,+1)
              else { aoff = E_BYTES + r * 2 * S_B + hf * 8 * 128; lbo = S_B; }                     // (0, 0) | unused
            }
            const uint32_t d = tmem + j * 128;
            const uint32_t acc = (it == 0 && r == 0 && hf == 0) ? 0u : 1u;
            if (X3) {
              umma_tf32(d, mn_desc(a_hi + aoff, lbo), bd, kIdesc128x128, acc, leader);
              umma_tf32(d + 64, mn_desc(a_lo + aoff, lbo), bd, kIdesc128x64, 1u, leader);
            } else {
              umma_tf32(d, mn_desc(a_hi + aoff, lbo), bd, kIdesc128x64, acc, leader);
            }
          }
        }
      }
      umma_commit(s_empty + s, leader);
      if (tile + 1 == t_end) umma_commit(done, leader);
    }
  } else {
    long long it = 0;
    for (long long tile = t_begin; tile < t_end; ++tile, ++it) {
      const int s = (int)(it % NST);
      mbar_wait(t_full + s, (uint32_t)((it / NST) & 1));
      const uint32_t a_hi = smem_u32(smem + s * STAGE2);
      split_sweep<X3, ROLE == 0>(a_hi, A_PLANE, (ROLE == 0 ? A_PLANE : E_BYTES + Z_BYTES) / 16, a_hi + 2 * A_PLANE, RT2, tid, dbs);
      fence_proxy_async();
      mbar_arrive_(s_full + s);
    }
  }
  mbar_wait(done, 0);
  tc_fence_after();
  __syncthreads();
  if (ROLE == 0 && a.part_db) {
    float* red = reinterpret_cast<float*>(smem);
    if (tid < kSplitThreads) {
      int channel, slot;
      db_slot(tid, channel, slot);
      *reinterpret_cast<float4*>(red + slot * 64 + channel) = dbs;
    }
    __syncthreads();
    if (tid < 64) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) t += red[r * 64 + tid];
      a.part_db[(long long)chunk * 64 + tid] = t;
    }
  }
  if (warp >= 8) return;
  const int q = warp & 3, half = warp >> 2, second = q >> 1, ci = (q & 1) * 32 + lane;
#pragma unroll 1
  for (int j = 0; j < NPAIR; ++j) {
    int tap;
    if (ROLE == 0) tap = second ? 6 + j : j;                    // (dy = +1 | -1, dx = j - 1)
    else tap = j == 0 ? (second ? 5 : 3) : (second ? -1 : 4);   // (0, +1 | -1)  |  (0, 0)
    uint32_t r0[32], r1[32];
    const uint32_t ta = tmem + (static_cast<uint32_t>(q * 32) << 16) + j * 128 + half * 32;
    tmem_ld32(ta, r0);
    if (X3) tmem_ld32(ta + 64, r1);
    if (tap >= 0) {
      float* po = a.part + ((long long)chunk * a.ntaps + tap) * 64 * 64 + ci;
#pragma unroll
      for (int i = 0; i < 32; ++i)
        po[(half * 32 + i) * 64] = (X3 ? __uint_as_float(r1[i]) : 0.f) + __uint_as_float(r0[i]);
    }
  }
}

template <bool X3>
__global__ void __launch_bounds__(kThreads, 1) tapwgrad_halo_s2_kernel(const HaloWgradArgs a,
                                                                        const __grid_constant__ HaloWgradS2Tma tm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + s2::NST * s2::STAGE2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * s2::NST + 2);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < s2::NST; ++s) {
      mbar_init(bars + s, 1);
      mbar_init(bars + s2::NST + s, kSplitThreads);
      mbar_init(bars + 2 * s2::NST + s, 1);
    }
    mbar_init(bars + 3 * s2::NST, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (blockIdx.y == 0) run_role_s2<X3, 0>(a, tm, smem, bars, tmem);
  else run_role_s2<X3, 1>(a, tm, smem, bars, tmem);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

template <bool X3>
int launch_s2(const HaloWgradArgs& h, int chunks, cudaStream_t st) {
  HaloWgradS2Tma tm;
  const uint64_t W = (uint64_t)h.W, H = (uint64_t)h.H, N = (uint64_t)h.N;   // dY geometry; x is [N, 2H, 2W, 64]
  const uint64_t dims[4] = {64, W, H, N};
  const uint64_t sy[3] = {256, W * 256, H * W * 256};
  const uint64_t sx[3] = {512, 2 * (2 * W) * 256, (2 * H) * (2 * W) * 256};
  const uint32_t box18[4] = {32, HW, 1, 1}, box16[4] = {32, TW, 1, 1};
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px)
      if (!tma::encode_f32_4d(&tm.x[py * 2 + px], h.x + ((long long)py * 2 * h.W + px) * 64, dims, sx,
                              (py == 1 && px == 1) ? box18 : box16, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B))
        return B200NP_E_UNSUPPORTED;
  if (!tma::encode_f32_4d(&tm.dy, h.dy, dims, sy, box16, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return B200NP_E_UNSUPPORTED;
  const size_t smem = s2::NST * s2::STAGE2 + 1024 + 1024;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(tapwgrad_halo_s2_kernel<X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return B200NP_E_LAUNCH;
    configured = true;
  }
  tapwgrad_halo_s2_kernel<X3><<<dim3(chunks, 2), kThreads, smem, st>>>(h, tm);
  return launch_status();
}

template <bool X3>
int launch_tma(const HaloWgradArgs& h, int chunks, cudaStream_t st) {
  HaloWgradTma tm;
  const uint64_t W = (uint64_t)h.W, H = (uint64_t)h.H, N = (uint64_t)h.N;
  const uint64_t dims[4] = {64, W, H, N};
  const uint64_t strides[3] = {256, W * 256, H * W * 256};
  const uint32_t box_x[4] = {32, HW, 1, 1}, box_y[4] = {32, TW, 1, 1};
  if (!tma::encode_f32_4d(&tm.x, h.x, dims, strides, box_x, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return B200NP_E_UNSUPPORTED;
  if (!tma::encode_f32_4d(&tm.dy, h.dy, dims, strides, box_y, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return B200NP_E_UNSUPPORTED;
  if (h.xs) {   // xs[2 y][2 x]: the parity-(0,0) view of [N, 2H, 2W, 64]
    const uint64_t s2[3] = {512, 2 * (2 * W) * 256, (2 * H) * (2 * W) * 256};
    if (!tma::encode_f32_4d(&tm.xs, h.xs, dims, s2, box_y, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return B200NP_E_UNSUPPORTED;
  } else {
    tm.xs = tm.dy;   // never dereferenced meaningfully: role 1 then multiplies the zeroed skip blocks
  }
  const size_t smem = 2 * STAGE + 1024 + 1024;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(tapwgrad_halo_tma_kernel<X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return B200NP_E_LAUNCH;
    configured = true;
  }
  tapwgrad_halo_tma_kernel<X3><<<dim3(chunks, 2), kThreads, smem, st>>>(h, tm);
  return launch_status();
}

}  // namespace

// Pixel chunks (= partial tiles per tap) of the halo formulation for an [N, OH, OW] output; 0 if the shape does not fit.
int tapwgrad_halo_chunks(int N, int OH, int OW) {
  if (N <= 0 || OH % RT || OW % TW) return 0;
  const long long tiles = (long long)N * (OH / RT) * (OW / TW);
  const long long per = ceil_div(tiles, kNumSMs);
  return (int)ceil_div(tiles, per);
}

// Stride-2 variant: tiles of 2 x 16 output pixels.
int tapwgrad_halo_s2_chunks(int N, int OH, int OW) {
  if (N <= 0 || OH % s2::RT2 || OW % TW) return 0;
  const long long tiles = (long long)N * (OH / s2::RT2) * (OW / TW);
  const long long per = ceil_div(tiles, kNumSMs);
  return (int)ceil_div(tiles, per);
}
static int launch_tapwgrad_halo_s2(TapWgradArgs& a, int precision, cudaStream_t st) {
  if (a.ntaps != 9 || a.srcH != 2 * a.OH || a.srcW != 2 * a.OW) return B200NP_E_UNSUPPORTED;
  for (int t = 0; t < 9; ++t)
    if (a.taps[t].src != 0 || a.taps[t].dy != t / 3 - 1 || a.taps[t].dx != t % 3 - 1) return B200NP_E_UNSUPPORTED;
  const int chunks = tapwgrad_halo_s2_chunks(a.N, a.OH, a.OW);
  if (chunks <= 0) return B200NP_E_UNSUPPORTED;
  HaloWgradArgs h{};
  h.x = a.src; h.dy = a.dy; h.xs = nullptr;
  h.part = a.part; h.part_db = a.part_db;
  h.N = a.N; h.H = a.OH; h.W = a.OW; h.ntaps = 9;
  h.tiles = (long long)a.N * (a.OH / s2::RT2) * (a.OW / TW);
  h.per = ceil_div(h.tiles, kNumSMs);
  const int rc = precision == B200NP_PREC_TF32 ? launch_s2<false>(h, chunks, st) : launch_s2<true>(h, chunks, st);
  if (rc == B200NP_OK) a.chunks = chunks;
  return rc;
}

// 3x3 stride-1 taps in row-major order (+ one skip tap on src2 with stride 2), or plain 3x3 stride 2; fills a.chunks
int launch_tapwgrad_halo(TapWgradArgs& a, int precision, cudaStream_t st) {
  if (precision == B200NP_PREC_FP32_SIMT || a.Cin != 64 || a.Cout != 64) return B200NP_E_UNSUPPORTED;
  if (a.in_s == 2) return launch_tapwgrad_halo_s2(a, precision, st);
  if (a.in_s != 1) return B200NP_E_UNSUPPORTED;
  if (a.ntaps != 9 && a.ntaps != 10) return B200NP_E_UNSUPPORTED;
  for (int t = 0; t < 9; ++t)
    if (a.taps[t].src != 0 || a.taps[t].dy != t / 3 - 1 || a.taps[t].dx != t % 3 - 1) return B200NP_E_UNSUPPORTED;
  if (a.ntaps == 10 && (a.taps[9].src != 1 || a.in_s2 != 2 || !a.src2 || a.src2H != 2 * a.OH || a.src2W != 2 * a.OW))
    return B200NP_E_UNSUPPORTED;
  const int chunks = tapwgrad_halo_chunks(a.N, a.OH, a.OW);
  if (chunks <= 0) return B200NP_E_UNSUPPORTED;
  HaloWgradArgs h{};
  h.x = a.src; h.dy = a.dy; h.xs = a.ntaps == 10 ? a.src2 : nullptr;
  h.part = a.part; h.part_db = a.part_db;
  h.N = a.N; h.H = a.OH; h.W = a.OW; h.ntaps = a.ntaps;
  h.tiles = (long long)a.N * (a.OH / RT) * (a.OW / TW);
  h.per = ceil_div(h.tiles, kNumSMs);
  const int rc = precision == B200NP_PREC_TF32 ? launch_tma<false>(h, chunks, st) : launch_tma<true>(h, chunks, st);
  if (rc == B200NP_OK) a.chunks = chunks;
  return rc;
}

}  // namespace b200np