// Halo-tile tcgen05 implementation of the tap convolution: forward 3x3 s1 (+ fused 1x1 s2 skip
// projection), forward 3x3 s2, data gradient of a 3x3 s1 conv, and the four parity classes of a
// stride-2 data gradient (+ skip gradient).
//
// Why: the gather kernel (tapconv_umma.cu) re-reads and re-splits every input pixel once per tap (9x) and
// is bound by the latency of those loads (ncu: long_scoreboard, tensor pipe 14 %).  Here an output tile is
// 16 rows x 8 pixels of one image; the input pixels it needs are loaded, split into tf32 hi/lo and stored
// in shared memory ONCE per 32-channel half, as one or more PLANES in the K-major SWIZZLE_128B layout with
// one 128-byte "slot" per pixel:
//   * a plane is a dense (16+dy_span) x (8+dx_span) window of one source tensor sampled at stride `scale`
//     with phase (py, px).  Stride-1 stencils need one plane (the halo).  A stride-2 forward conv needs the
//     four parity planes x[2i+py, 2j+px]: in each of them consecutive OUTPUT pixels are consecutive slots.
//     The fused skip projection / skip gradient is one more plane (16 x 8, no halo).
//   * a tap is then nothing but a descriptor: start = slot(plane, dy, dx), 8 consecutive slots = 8
//     consecutive output pixels, stride between the 16 row groups (SBO) = plane pitch * 128 B.
//     (The tensor core applies the 128B swizzle to absolute shared-memory address bits, so start addresses
//     at any 128-byte slot and any SBO are legal as long as the data is stored with the same
//     absolute-address swizzle -- verified on B200 by tools/probe.)
//
// Weights arrive pre-split (hi/lo) and pre-swizzled from b200np_pack_conv_weight, one 16 KB K-block
// (tap, channel half) per cp.async.bulk into a ring of 3, 4 or 6 slots.
//
// Persistent, warp-specialised CTA (one per SM), tiles round-robin, one stage = one channel half of one tile:
//   warp  14    plane loader: ONE cp.async.bulk.tensor per plane (HaloTma) lands the raw fp32 pixels in the `hi`
//               plane of the stage -- no global-load / address arithmetic in any thread, out-of-bounds pixels
//               zero-filled by the copy engine;
//   warps 0-7   split warps: shared memory -> shared memory, one LDS + one STS per 16 bytes.  fp32-grade mode: the
//               landed raw plane is used as the `hi` operand as it is -- the tensor core truncates fp32 to tf32 --
//               and only lo = x - trunc_tf32(x) is written to the `lo` plane; single-pass mode: the landed values
//               are rounded to nearest in place.  (Producers that gathered with global loads spent LDG + address
//               decode + two STS per 16 bytes; the L1 data pipe, which the tensor core's operand reads share, was
//               95 % busy: 0.57 ms against 0.535 ms on the layer1 conv2 + skip launch.)
//   warp  8     weight loader (one lane issues bulk copies); also owns the TMEM allocation
//   warp  9     MMA issuer with the tap loop unrolled (9 or 10 taps): every per-tap descriptor word is a
//               loop-invariant uniform register, and the `weights landed` probe of tap t+1 is issued before the
//               MMAs of tap t, so its ~90-cycle latency hides behind the issue of eight MMAs
//   warps 10-13 epilogue (TMEM -> registers -> bias / ReLU mask / activation -> NHWC global)
// Two accumulator sets in TMEM let the epilogue of tile i overlap the MMAs of tile i+1.
//
// fp32-grade mode: N = 64 tf32 MMAs are shared-memory-bandwidth bound (54.5 cycles instead of 32,
// tools/probe/probe_mma_rate.cu), so the weight slot [B_hi ; B_lo] is used as ONE 128-row operand:
// A_hi x [B_hi;B_lo] (N = 128, 64 cycles) yields hi*hi (columns 0-63) and hi*lo (64-127), then A_lo x B_hi
// (N = 64) adds the other cross term into columns 64-127.  Accumulator blocks of 128 columns rotate (kRot)
// to bound the bias of the tensor core's truncating fp32 accumulation; the epilogue sums them.

#include "tapconv.cuh"
#include "tma.cuh"
#include "umma.cuh"

namespace b200np {

using namespace umma;

namespace {

constexpr int kTileRows = 16, kTileCols = 8;
constexpr int kMaxPlanes = 5;
constexpr int kMaxBStages = 6;                           // deepest weight ring (launch_halo picks 3, 4 or 6)
constexpr int kRot = 2;                                  // rotating accumulator blocks per accumulator set
constexpr uint32_t kBSlotBytes = 2 * kBBytes;            // hi + lo = 16 KB
constexpr int kSplitWarps = 8, kSplitThreads = 32 * kSplitWarps;
constexpr int kWeightWarp = 8, kMmaWarp = 9, kEpiWarp0 = 10, kTmaWarp = 14;
constexpr int kThreads = 32 * (kTmaWarp + 1);
constexpr uint32_t kSmemBudget = 227 * 1024;

struct Plane {
  const float* src;     // NHWC tensor [N, srcH, srcW, 64]
  int srcH, srcW;
  int scale, py, px;    // source pixel = ((oy0 + dy_min + hy) * scale + py, (ox0 + dx_min + hx) * scale + px)
  int dy_min, dx_min, HR, HC;
  int slot0, nslots;    // slots [slot0, slot0 + nslots) of the stage; both multiples of 8
};

struct HaloArgs {
  TapConvArgs t;        // epilogue fields, tap list (src / slab), output geometry
  const float* bp[2];   // pre-split, pre-swizzled weights per source: [half][slab][hi 8 KB | lo 8 KB]
  int nslabs[2];
  int nplanes;
  Plane pl[kMaxPlanes];
  int tap_off[kMaxTaps];   // first slot of the tap's window inside the stage
  int tap_hc[kMaxTaps];    // pitch (slots per plane row) of the tap's plane
  int total_slots;         // per stage plane
  int ncls;                // 1, or the number of output classes (TapClasses): one accumulator set per class
  int tap_cls[kMaxTaps];
  int cls_oy[4], cls_ox[4];
  int a_stages;            // 1 or 2 plane stages
  int tiles_x, tiles_total;
  uint32_t plane_bytes, stage_bytes, b_off, bar_off;
  int nb;                  // weight ring depth
};

// Tensor maps of the planes: one 4-D map per plane over its source tensor -- [channel][x][y][image],
// for a stride-2 parity plane the view x[2j + px][2i + py] (base shifted, strides doubled) -- with a box of 32 channels
// x HC x HR x 1 and SWIZZLE_128B, so that ONE bulk tensor copy lands a whole plane of a channel half in exactly the
// slot layout the UMMA descriptors expect; out-of-bounds pixels arrive as zeros (= the convolution's padding).
struct HaloTma {
  tma::Map plane[kMaxPlanes];
};

template <bool X3>
constexpr uint32_t b_slot_bytes() { return X3 ? kBSlotBytes : kBBytes; }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

struct Ring {
  int idx = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance(int n) {
    if (++idx == n) { idx = 0; phase ^= 1; }
  }
};

// ===================== epilogue =====================
// warps kEpiWarp0 .. kEpiWarp0+3: TMEM -> registers -> bias / ReLU gates / activation -> NHWC global
template <bool X3>
__device__ __forceinline__ void halo_epilogue(const HaloArgs& h, uint64_t* acc_full, uint64_t* acc_empty,
                                              uint32_t tmem_base, int warp, int lane) {
  const TapConvArgs& a = h.t;
  constexpr uint32_t kAccCols = X3 ? 256u : 128u;
  constexpr uint32_t kBlkCols = X3 ? 128u : 64u;
  const int ncls = h.ncls, ntaps = a.ntaps;
  const uint32_t set_stride = ncls > 1 ? kBlkCols : kAccCols;
  // ===================== epilogue =====================
  // (A shared-memory transposed store, which halved the stem kernel's time, was measured here and made this
  // kernel slower -- 1.16 -> 2.3 ms for the fused stride-2 data gradient: with one epilogue warp per scheduler
  // the extra STS/LDS/__syncwarp round trip is pure latency.  Direct 16-byte stores per pixel row are kept.)
  const int q = warp & 3;                              // TMEM lane quarter this warp may access (warp id % 4)
  const int m = q * 32 + lane;                         // accumulator row = output pixel of the tile
  int acc_set = 0;
  uint32_t acc_phase = 0;
  const int kb_total = 2 * ntaps;
  const int blocks_used = ncls > 1 ? 1 : (kb_total < kRot ? kb_total : kRot);
  for (int tile = blockIdx.x; tile < h.tiles_total; tile += gridDim.x) {
    const int xt = tile % h.tiles_x, rb = tile / h.tiles_x;
    const int r0 = rb * kTileRows;
    const int n = r0 / a.OH, oy = r0 - n * a.OH + (m >> 3), ox = xt * kTileCols + (m & 7);
    // The packed ReLU gates of this thread's pixels (all classes) are fetched BEFORE the accumulators are waited
    // for: with one epilogue warp per scheduler a load issued after the wait is pure exposed latency, and that
    // latency (8 dependent mask loads per tile) was what paced the fused stride-2 data gradient.
    uint32_t mw[4][2] = {};
    if (a.mask_bits) {
#pragma unroll
      for (int cc = 0; cc < 4; ++cc)
        if (cc < ncls) {
          const int d_oy = ncls > 1 ? h.cls_oy[cc] : a.dst_oy, d_ox = ncls > 1 ? h.cls_ox[cc] : a.dst_ox;
          const long long px = ((long long)n * a.dstH + (long long)oy * a.dst_s + d_oy) * a.dstW + (long long)ox * a.dst_s + d_ox;
          const uint2 w2 = __ldg(reinterpret_cast<const uint2*>(a.mask_bits + px * 2));
          mw[cc][0] = w2.x; mw[cc][1] = w2.y;
        }
    }
   for (int cls = 0; cls < ncls; ++cls) {               // class mode: the tile's outputs, one accumulator set each
    // (not unrolled: four copies of the epilogue body thrash the instruction cache; the prefetched gate words
    // are picked with selects instead of register indexing)
    const uint32_t mw0 = cls == 0 ? mw[0][0] : cls == 1 ? mw[1][0] : cls == 2 ? mw[2][0] : mw[3][0];
    const uint32_t mw1 = cls == 0 ? mw[0][1] : cls == 1 ? mw[1][1] : cls == 2 ? mw[2][1] : mw[3][1];
    const int set = ncls > 1 ? cls : acc_set;
    const int d_oy = ncls > 1 ? h.cls_oy[cls] : a.dst_oy, d_ox = ncls > 1 ? h.cls_ox[cls] : a.dst_ox;
    const long long off =
        (((long long)n * a.dstH + (long long)oy * a.dst_s + d_oy) * a.dstW + (long long)ox * a.dst_s + d_ox) * 64;
    mbar_wait(acc_full + set, acc_phase);
    tc_fence_after();
    const uint32_t taddr = tmem_base + set * set_stride + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      float acc[32];
      {   // sum the rotating blocks (and, fp32-grade, their cross-term column group), smallest terms first
        uint32_t r[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0.f;
        if (X3) {
#pragma unroll
          for (int b = 0; b < kRot; ++b)
            if (b < blocks_used) {
              tmem_ld32(taddr + b * 128 + 64 + hf * 32, r);
#pragma unroll
              for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r[j]);
            }
        }
#pragma unroll
        for (int b = 0; b < kRot; ++b)
          if (b < blocks_used) {
            tmem_ld32(taddr + b * (X3 ? 128 : 64) + hf * 32, r);
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r[j]);
          }
      }
      if (hf == 1) {                                   // all TMEM reads of this set are done
        tc_fence_before();
        mbar_arrive(acc_empty + set);
      }
      const uint32_t mword = hf ? mw1 : mw0;             // 32 ReLU gates
      uint32_t gates = 0u;                               // (output > 0) of this thread's 32 channels
      // float-mask variant: all eight loads are issued before the first use (one exposed latency, not eight)
      const bool fmask = !a.mask_bits && a.mask;
      float4 mk8[8];
      if (fmask) {
#pragma unroll
        for (int qq = 0; qq < 8; ++qq) mk8[qq] = ldg4(a.mask + off + hf * 32 + 4 * qq);
      }
#pragma unroll
      for (int qq = 0; qq < 8; ++qq) {
        const int c = hf * 32 + 4 * qq;
        float4 o = make_float4(acc[4 * qq], acc[4 * qq + 1], acc[4 * qq + 2], acc[4 * qq + 3]);
        if (a.bias) {
          const float4 b = ldg4(a.bias + c);
          o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
        }
        if (a.bias2) {
          const float4 b = ldg4(a.bias2 + c);
          o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
        }
        if (a.mask_bits) {
          const uint32_t nb4 = mword >> (4 * qq);
          o.x = (nb4 & 1u) ? o.x : 0.f; o.y = (nb4 & 2u) ? o.y : 0.f;
          o.z = (nb4 & 4u) ? o.z : 0.f; o.w = (nb4 & 8u) ? o.w : 0.f;
        } else if (fmask) {
          const float4 mk = mk8[qq];
          o.x = mk.x > 0.f ? o.x : 0.f; o.y = mk.y > 0.f ? o.y : 0.f;
          o.z = mk.z > 0.f ? o.z : 0.f; o.w = mk.w > 0.f ? o.w : 0.f;
        }
        if (a.act == B200NP_ACT_RELU) {
          o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
        }
        *reinterpret_cast<float4*>(a.dst + off + c) = o;
        gates |= (uint32_t)((o.x > 0.f) | ((o.y > 0.f) << 1) | ((o.z > 0.f) << 2) | ((o.w > 0.f) << 3)) << (4 * qq);
      }
      if (a.relu_bits) a.relu_bits[(off >> 6) * 2 + hf] = gates;
    }
   }
    if (ncls > 1) acc_phase ^= 1;                      // every class set is used once per tile
    else if (++acc_set == 2) { acc_set = 0; acc_phase ^= 1; }
  }
}

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

template <bool X3, int NT, int NB>
__global__ void __launch_bounds__(kThreads, 1) tapconv_halo_tma_kernel(const HaloArgs h, const __grid_constant__ HaloTma tm) {
  constexpr uint32_t kBSlot = b_slot_bytes<X3>();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + h.bar_off);
  uint64_t* a_full = bars;                  // [a_stages] split warps -> MMA          (count 256)
  uint64_t* a_empty = bars + 2;             // [a_stages] MMA commit -> plane loader  (count 1)
  uint64_t* acc_full = bars + 4;            // [4] MMA commit -> epilogue             (count 1)
  uint64_t* acc_empty = bars + 8;           // [4] epilogue -> MMA                    (count 128)
  uint64_t* b_full = bars + 12;             // [nb] bulk copy tx -> MMA               (count 1 + tx)
  uint64_t* b_empty = b_full + kMaxBStages; // [nb] MMA commit -> weight warp         (count 1)
  uint64_t* t_full = b_empty + kMaxBStages; // [a_stages] tensor copies tx -> split warps, MMA (count 1 + tx)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_full + 2);
  const int nb = h.nb, a_stages = h.a_stages;

  const TapConvArgs& a = h.t;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr uint32_t kAccCols = X3 ? 256u : 128u;
  constexpr uint32_t kTmemCols = 2 * kAccCols;
  constexpr uint32_t kBlkCols = X3 ? 128u : 64u;
  const int ncls = h.ncls;

  if (tid == 0) {
    for (int s = 0; s < a_stages; ++s) {
      mbar_init(a_full + s, kSplitThreads);
      mbar_init(a_empty + s, 1);
      mbar_init(t_full + s, 1);
    }
    for (int s = 0; s < nb; ++s) { mbar_init(b_full + s, 1); mbar_init(b_empty + s, 1); }
    for (int s = 0; s < 4; ++s) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kWeightWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == kTmaWarp && lane == 0) {
    for (int p = 0; p < h.nplanes; ++p) tma::prefetch_map(&tm.plane[p]);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kSplitWarps) {
    // ===================== split warps: smem -> smem =====================
    Ring st;
    const uint32_t units = (uint32_t)h.total_slots * 8u;      // 16-byte units of one plane copy
    for (int tile = blockIdx.x; tile < h.tiles_total; tile += gridDim.x)
      for (int half = 0; half < 2; ++half) {
        mbar_wait(t_full + st.idx, st.phase);                  // the tensor copies of this stage have landed
        const uint32_t hi = smem_u32(smem + st.idx * h.stage_bytes), lo = hi + h.plane_bytes;
        for (uint32_t u0 = tid; u0 < units; u0 += 4 * kSplitThreads) {
          float4 v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t u = u0 + j * kSplitThreads;
            if (u < units) v[j] = lds128(hi + u * 16u);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t u = u0 + j * kSplitThreads;
            if (u < units) {
              if (X3) sts128(lo + u * 16u, lo_of_truncated(v[j]));   // the raw plane is the hi operand (hardware truncation)
              else sts128(hi + u * 16u, to_tf32_4(v[j]));            // single pass: round to nearest in place
            }
          }
        }
        fence_proxy_async();
        mbar_arrive(a_full + st.idx);
        st.advance(a_stages);
      }
  } else if (warp == kTmaWarp) {
    // ===================== plane loader (TMA) =====================
    const uint32_t leader = elect_one_sync();
    Ring st;
    uint32_t stage_tx = 0;
    for (int p = 0; p < h.nplanes; ++p) stage_tx += (uint32_t)(h.pl[p].HR * h.pl[p].HC) * 128u;
    for (int tile = blockIdx.x; tile < h.tiles_total; tile += gridDim.x) {
      const int xt = tile % h.tiles_x, rb = tile / h.tiles_x;
      const int r0 = rb * kTileRows;
      const int n = r0 / a.OH, oy0 = r0 - n * a.OH, ox0 = xt * kTileCols;
      for (int half = 0; half < 2; ++half) {
        mbar_wait(a_empty + st.idx, st.phase ^ 1);             // the MMAs that read this stage have retired
        if (leader) mbar_expect_tx(t_full + st.idx, stage_tx);
        const uint32_t stage = smem_u32(smem + st.idx * h.stage_bytes);
        for (int p = 0; p < h.nplanes; ++p)
          tma::load_4d(stage + (uint32_t)h.pl[p].slot0 * 128u, &tm.plane[p], smem_u32(t_full + st.idx), half * 32,
                       ox0 + h.pl[p].dx_min, oy0 + h.pl[p].dy_min, n, leader);
        st.advance(a_stages);
      }
    }
  } else if (warp == kWeightWarp) {
    // ===================== weight loader =====================
    const bool leader = elect_one_sync();
    Ring bs;
    for (int tile = blockIdx.x; tile < h.tiles_total; tile += gridDim.x)
      for (int half = 0; half < 2; ++half)
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          const Tap tp = a.taps[t];
          const float* src = h.bp[tp.src] + ((long long)half * h.nslabs[tp.src] + tp.slab) * (kBSlotBytes / 4);
          mbar_wait(b_empty + bs.idx, bs.phase ^ 1);
          if (leader) {
            mbar_expect_tx(b_full + bs.idx, kBSlot);
            bulk_g2s(smem + h.b_off + bs.idx * kBSlot, src, kBSlot, b_full + bs.idx);
          }
          bs.advance(nb);
        }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    // Work elimination on the kernel's first form (profiles/halo_stalls_r1.txt) showed MMAs + handshakes alone at
    // 0.51 of 0.57 ms and the handshake skeleton WITHOUT any MMA at 8.4 K cycles per tile: the issuing lane's own
    // ~100 instructions per K-block (constant-bank loads, R2UR moves, ring arithmetic, a 90-cycle barrier probe) do
    // not overlap the 474 tensor cycles of the K-block, because the tensor queue is shallow.  So here everything that
    // can be is a compile-time constant: taps and halves are unrolled, the weight ring depth NB divides the 2*NT
    // K-blocks of a tile (slot index and phase parity of every K-block are literals), per-tap descriptor words are
    // loop-invariant registers, the whole warp runs the loop uniformly and only tcgen05.mma / tcgen05.commit carry the
    // elected-lane predicate (no divergent region, no R2UR), and the probe of the next weight slot is issued before
    // the current tap's MMAs.
    static_assert((2 * NT) % NB == 0, "ring depth must divide the K-blocks of a tile");
    constexpr uint32_t kWraps = 2 * NT / NB;                 // ring passes per tile
    const uint32_t leader = elect_one_sync();
    int acc_set = 0;
    uint32_t acc_phase = 0, cphase = 0;
    const uint32_t plane16 = h.plane_bytes >> 4;
    const uint32_t lbo_bits = 1u << 16;
    const uint32_t b_hi_word = (1024u >> 4) | (1u << 14) | (2u << 29);
    const uint32_t b_base16 = ((smem_u32(smem + h.b_off) & 0x3FFFFu) >> 4) | lbo_bits;
    const uint32_t smem16 = (smem_u32(smem) & 0x3FFFFu) >> 4;
    const uint32_t stage16_step = h.stage_bytes >> 4;
    const uint32_t b_full_a = smem_u32(b_full), b_empty_a = smem_u32(b_empty);
    constexpr uint32_t kIdescN128 = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    uint32_t a_off16[NT], a_hiw[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      a_off16[t] = (uint32_t)h.tap_off[t] * 8u;
      a_hiw[t] = (((uint32_t)h.tap_hc[t] * 128u) >> 4) | (1u << 14) | (2u << 29);   // SBO, version 1, SWIZZLE_128B
    }
    auto mma = [&](uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t acc, uint32_t idesc) {
      asm volatile(
          "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
          "mov.b64 da, {%1, %2};\n\t"
          "mov.b64 db, {%3, %4};\n\t"
          "setp.ne.b32 p, %6, 0;\n\t"
          "setp.ne.b32 q, %7, 0;\n\t"
          "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
          ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi_word), "r"(idesc), "r"(acc), "r"(leader)
          : "memory");
    };
    auto commit_a = [&](uint32_t bar_addr) {
      asm volatile(
          "{\n\t.reg .pred q;\n\t"
          "setp.ne.b32 q, %1, 0;\n\t"
          "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
          ::"r"(bar_addr), "r"(leader)
          : "memory");
    };
    auto probe = [&](uint32_t bar_addr, uint32_t parity) -> bool {
      uint32_t ok;
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(ok)
          : "r"(bar_addr), "r"(parity)
          : "memory");
      return ok != 0;
    };
    bool b_ready = false;                                    // answer of the early probe of the next weight slot
    uint32_t it = 0;                                         // tiles this CTA has processed
    for (int tile = blockIdx.x; tile < h.tiles_total; tile += gridDim.x, ++it) {
      if (ncls == 1) {
        mbar_wait(acc_empty + acc_set, acc_phase ^ 1);       // the epilogue has drained this set
        tc_fence_after();
      }
      const uint32_t d0 = tmem_base + acc_set * kAccCols;
      const uint32_t ring_par0 = it * kWraps;                // ring passes completed before this tile
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const uint32_t sidx = a_stages == 2 ? (uint32_t)half : 0u;
        const uint32_t spar = a_stages == 2 ? (it & 1u) : ((2u * it + half) & 1u);
        mbar_wait(t_full + sidx, spar);                      // hi plane landed (async proxy) ...
        mbar_wait(a_full + sidx, spar);                      // ... and was rounded / split by the split warps
        const uint32_t stage16 = (smem16 + sidx * stage16_step) | lbo_bits;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          constexpr int dummy = 0; (void)dummy;
          const int kb = half * NT + t;                      // literal after unrolling
          const uint32_t slot = (uint32_t)(kb % NB), pass = (uint32_t)(kb / NB);
          const uint32_t kbn = (uint32_t)((kb + 1) % (2 * NT));
          const uint32_t slot_n = kbn % NB, pass_n = kbn / NB + (kb + 1 == 2 * NT ? kWraps : 0u);
          if (!b_ready) mbar_wait(b_full + slot, (ring_par0 + pass) & 1u);
          b_ready = probe(b_full_a + slot_n * 8u, (ring_par0 + pass_n) & 1u);   // next slot: answer used after these MMAs
          const uint32_t ah = stage16 + a_off16[t], al = ah + plane16;
          const uint32_t bh = b_base16 + slot * (kBSlot >> 4);
          uint32_t d_blk = d0 + (uint32_t)(kb % kRot) * kBlkCols;
          uint32_t acc_first = kb >= kRot;
          int cls = 0;
          bool cls_last = false;
          if (ncls > 1) {
            cls = h.tap_cls[t];
            const bool cls_first = t == 0 || h.tap_cls[t > 0 ? t - 1 : 0] != cls;
            cls_last = t == NT - 1 || h.tap_cls[t < NT - 1 ? t + 1 : t] != cls;
            if (half == 0 && cls_first) {                    // the epilogue has drained this class of the previous tile
              mbar_wait(acc_empty + cls, cphase ^ 1);
              tc_fence_after();
            }
            d_blk = tmem_base + cls * kBlkCols;
            acc_first = !(half == 0 && cls_first);
          }
          if (X3) {
#pragma unroll
            for (int k = 0; k < 4; ++k) mma(d_blk, ah + 2 * k, a_hiw[t], bh + 2 * k, k == 0 ? acc_first : 1u, kIdescN128);
#pragma unroll
            for (int k = 0; k < 4; ++k) mma(d_blk + 64, al + 2 * k, a_hiw[t], bh + 2 * k, 1u, kIdescTf32_128x64);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) mma(d_blk, ah + 2 * k, a_hiw[t], bh + 2 * k, k == 0 ? acc_first : 1u, kIdescTf32_128x64);
          }
          commit_a(b_empty_a + slot * 8u);
          if (ncls > 1 && half == 1 && cls_last) umma_commit(acc_full + cls, leader);   // class complete
        }
        umma_commit(a_empty + sidx, leader);
      }
      if (ncls == 1) {
        umma_commit(acc_full + acc_set, leader);
        if (++acc_set == 2) { acc_set = 0; acc_phase ^= 1; }
      } else {
        cphase ^= 1;
      }
    }
  } else if (warp >= kEpiWarp0 && warp < kEpiWarp0 + 4) {
    halo_epilogue<X3>(h, acc_full, acc_empty, tmem_base, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWeightWarp) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

template <bool X3, int NT, int NB>
int launch_halo_tma_t(const HaloArgs& h, const HaloTma& tm, size_t smem, cudaStream_t st) {
  static size_t configured = 0;
  if (smem > configured) {
    if (cudaFuncSetAttribute(tapconv_halo_tma_kernel<X3, NT, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)smem) != cudaSuccess)
      return B200NP_E_LAUNCH;
    configured = smem;
  }
  int grid = h.tiles_total < kNumSMs ? h.tiles_total : kNumSMs;
  tapconv_halo_tma_kernel<X3, NT, NB><<<grid, kThreads, smem, st>>>(h, tm);
  return launch_status();
}

// One tensor map per plane (see HaloTma).  false: some plane cannot be expressed (odd extent under a stride-2 view,
// driver without tensor-map support) -- the convolution then runs on the gather kernel.
static bool build_plane_maps(const HaloArgs& h, HaloTma& tm) {
  for (int p = 0; p < h.nplanes; ++p) {
    const Plane& P = h.pl[p];
    const uint64_t W = (uint64_t)P.srcW, H = (uint64_t)P.srcH, N = (uint64_t)h.t.N;
    const float* base = P.src;
    uint64_t dims[4] = {64, W, H, N};
    uint64_t strides[3] = {256, W * 256, H * W * 256};
    if (P.scale == 2) {
      if ((W | H) & 1) return false;
      base += ((long long)P.py * P.srcW + P.px) * 64;
      dims[1] = W / 2; dims[2] = H / 2;
      strides[0] = 512; strides[1] = 2 * W * 256;
    } else if (P.scale != 1) {
      return false;
    }
    const uint32_t box[4] = {32, (uint32_t)P.HC, (uint32_t)P.HR, 1};
    if (!tma::encode_f32_4d(&tm.plane[p], base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return false;
  }
  return true;
}

template <bool X3>
int launch_halo(HaloArgs& h, cudaStream_t st) {
  // shared-memory plan: one or two plane stages, then a weight ring whose depth divides the 2 * ntaps K-blocks of a
  // tile (the MMA issuer's slot indices are compile-time constants): 4 slots for 10 taps, 6 or 3 for 9
  const uint32_t planes = X3 ? 2u : 1u;
  h.plane_bytes = (uint32_t)h.total_slots * 128u;
  h.stage_bytes = planes * h.plane_bytes;
  const uint32_t tail = 1024 /*alignment slack*/ + 1024 /*barriers + plane table*/;
  const uint32_t bslot = b_slot_bytes<X3>();
  h.a_stages = (2 * h.stage_bytes + 2 * bslot + tail <= kSmemBudget) ? 2 : 1;
  if (h.a_stages * h.stage_bytes + 2 * bslot + tail > kSmemBudget) return B200NP_E_UNSUPPORTED;
  h.b_off = h.a_stages * h.stage_bytes;
  const int nb = (int)((kSmemBudget - tail - h.b_off) / bslot);
  const int want = h.t.ntaps == 10 ? 4 : (nb >= 6 ? 6 : 3);
  HaloTma tm;
  if (nb < want || !build_plane_maps(h, tm)) return B200NP_E_UNSUPPORTED;
  h.nb = want;
  h.bar_off = h.b_off + want * bslot;
  const size_t smem = h.bar_off + tail;
  if (h.t.ntaps == 10) return launch_halo_tma_t<X3, 10, 4>(h, tm, smem, st);
  return want == 6 ? launch_halo_tma_t<X3, 9, 6>(h, tm, smem, st) : launch_halo_tma_t<X3, 9, 3>(h, tm, smem, st);
}

}  // namespace

// Eligibility + geometry.  `bp0` / `bp1`: pre-split weights of source 0 / 1 (see b200np_pack_conv_weight).
int launch_tapconv_halo(const TapConvArgs& a, const float* bp0, int nslabs0, const float* bp1, int nslabs1,
                        int precision, cudaStream_t st, const TapClasses* cls) {
  // the MMA issuer unrolls the tap loop: 9 taps (3x3), or 10 (3x3 + the fused 1x1 skip)
  if (a.Cin != 64 || a.Cout != 64 || (a.ntaps != 9 && a.ntaps != 10) || !bp0) return B200NP_E_UNSUPPORTED;
  if (a.act != B200NP_ACT_NONE && a.act != B200NP_ACT_RELU) return B200NP_E_UNSUPPORTED;
  if (a.OH % kTileRows != 0 || a.OW % kTileCols != 0) return B200NP_E_UNSUPPORTED;
  if (a.in_s[0] != 1 && a.in_s[0] != 2) return B200NP_E_UNSUPPORTED;
  HaloArgs h{};
  h.t = a;
  h.ncls = 1;
  if (cls) {
    if (cls->ncls < 2 || cls->ncls > 4) return B200NP_E_UNSUPPORTED;
    h.ncls = cls->ncls;
    for (int t = 0; t < a.ntaps; ++t) {
      if (cls->tap_cls[t] < 0 || cls->tap_cls[t] >= cls->ncls || (t > 0 && cls->tap_cls[t] < cls->tap_cls[t - 1]))
        return B200NP_E_UNSUPPORTED;           // taps must be sorted by class
      h.tap_cls[t] = cls->tap_cls[t];
    }
    for (int c = 0; c < 4; ++c) { h.cls_oy[c] = cls->oy[c]; h.cls_ox[c] = cls->ox[c]; }
    for (int c = 0; c < cls->ncls; ++c) {      // every class needs at least one tap (its set is waited on per tile)
      bool any = false;
      for (int t = 0; t < a.ntaps; ++t) any |= cls->tap_cls[t] == c;
      if (!any) return B200NP_E_UNSUPPORTED;
    }
  }
  h.bp[0] = bp0; h.bp[1] = bp1; h.nslabs[0] = nslabs0; h.nslabs[1] = nslabs1;
  // group the taps into planes: (source, row parity, column parity) for a stride-2 source, one plane otherwise
  struct Key { int src, py, px; } keys[kMaxPlanes];
  int lo_y[kMaxPlanes], hi_y[kMaxPlanes], lo_x[kMaxPlanes], hi_x[kMaxPlanes];
  int tap_plane[kMaxTaps], tap_dy[kMaxTaps], tap_dx[kMaxTaps];
  int np = 0;
  for (int t = 0; t < a.ntaps; ++t) {
    const Tap& tp = a.taps[t];
    int py = 0, px = 0, dy = tp.dy, dx = tp.dx;
    if (tp.src == 1) {
      if (tp.dy != 0 || tp.dx != 0 || !bp1) return B200NP_E_UNSUPPORTED;
    } else if (a.in_s[0] == 2) {
      py = tp.dy & 1; px = tp.dx & 1;          // x[2o + d] = plane(d & 1)[o + (d - (d & 1)) / 2]
      dy = (tp.dy - py) / 2; dx = (tp.dx - px) / 2;
    }
    int p = 0;
    for (; p < np; ++p)
      if (keys[p].src == tp.src && keys[p].py == py && keys[p].px == px) break;
    if (p == np) {
      if (np == kMaxPlanes) return B200NP_E_UNSUPPORTED;
      keys[np] = Key{tp.src, py, px};
      lo_y[np] = hi_y[np] = dy; lo_x[np] = hi_x[np] = dx;
      ++np;
    } else {
      lo_y[p] = dy < lo_y[p] ? dy : lo_y[p]; hi_y[p] = dy > hi_y[p] ? dy : hi_y[p];
      lo_x[p] = dx < lo_x[p] ? dx : lo_x[p]; hi_x[p] = dx > hi_x[p] ? dx : hi_x[p];
    }
    tap_plane[t] = p; tap_dy[t] = dy; tap_dx[t] = dx;
  }
  int slot = 0;
  for (int p = 0; p < np; ++p) {
    Plane& P = h.pl[p];
    const int s = keys[p].src;
    P.src = a.src[s]; P.srcH = a.srcH[s]; P.srcW = a.srcW[s];
    P.scale = a.in_s[s]; P.py = keys[p].py; P.px = keys[p].px;
    P.dy_min = lo_y[p]; P.dx_min = lo_x[p];
    P.HR = kTileRows + hi_y[p] - lo_y[p]; P.HC = kTileCols + hi_x[p] - lo_x[p];
    if (P.HR > 255 || P.HC > 255) return B200NP_E_UNSUPPORTED;
    P.slot0 = slot; P.nslots = (P.HR * P.HC + 7) & ~7;
    slot += P.nslots;
  }
  h.nplanes = np;
  h.total_slots = slot;
  for (int t = 0; t < a.ntaps; ++t) {
    const Plane& P = h.pl[tap_plane[t]];
    h.tap_off[t] = P.slot0 + (tap_dy[t] - P.dy_min) * P.HC + (tap_dx[t] - P.dx_min);
    h.tap_hc[t] = P.HC;
  }
  h.tiles_x = a.OW / kTileCols;
  const long long tiles = (long long)a.N * a.OH / kTileRows * h.tiles_x;
  if (tiles <= 0) return B200NP_OK;
  if (tiles > 0x7fffffff) return B200NP_E_UNSUPPORTED;
  h.tiles_total = (int)tiles;
  return precision == B200NP_PREC_TF32 ? launch_halo<false>(h, st) : launch_halo<true>(h, st);
}

}  // namespace b200np
