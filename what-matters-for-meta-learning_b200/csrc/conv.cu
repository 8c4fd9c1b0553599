// C ABI of the channel-dense NHWC convolutions: builds tap tables (tapconv.cuh) for forward,
// data-gradient and weight-gradient and dispatches to the tcgen05 kernels (64-channel layers) or
// the CUDA-core kernels (fp32 validation mode; 32/48-channel layers of encoder_w0).
#include "tapconv.cuh"
#include "umma.cuh"

using namespace b200np;

namespace {

// Packed weight buffers (opaque to callers; size = b200np_packed_weight_floats):
//   [0, RR*Cout*Cin)            K-major slabs   wf: [t][co][ci]    wd: [t][ci][co]
//   64x64 layers only, after that: the tensor-core image of the same slabs, split into tf32 hi / lo and
//   laid out as ready-to-copy SWIZZLE_128B tiles  [half][t][hi 8 KB | lo 8 KB]  (row = output channel of
//   the GEMM, 32 reduction channels per row) -- one cp.async.bulk per K-block in tapconv_halo.cu.
__device__ __forceinline__ void put_umma(float* img, int RR, int t, int row, int k, float v) {
  const int half = k >> 5, c = (k & 31) >> 2, e = k & 3;
  const float hi = umma::to_tf32(v), lo = umma::to_tf32(v - hi);
  const long long tile = ((long long)half * RR + t) * 4096;          // floats per [hi|lo] K-block
  const int off = ((row >> 3) * 1024 + (row & 7) * 128 + ((c ^ (row & 7)) << 4)) / 4 + e;
  img[tile + off] = hi;
  img[tile + 2048 + off] = lo;
}
__global__ void pack_weight_kernel(const float* __restrict__ w, float* __restrict__ wf, float* __restrict__ wd,
                                   int Cout, int Cin, int RR, int umma_img) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int total = Cout * Cin * RR;
  if (i >= total) return;
  // torch layout: ((co*Cin + ci)*RR + t)
  int t = i % RR, r = i / RR;
  int ci = r % Cin, co = r / Cin;
  float v = w[i];
  if (wf) wf[((long long)t * Cout + co) * Cin + ci] = v;
  if (wd) wd[((long long)t * Cin + ci) * Cout + co] = v;
  if (umma_img) {
    if (wf) put_umma(wf + total, RR, t, co, ci, v);
    if (wd) put_umma(wd + total, RR, t, ci, co, v);
  }
}

// Pixel chunks per weight gradient.  The tcgen05 kernel runs one CTA per (tap pair, chunk), two CTAs
// per SM: size the grid to full waves (a ragged last wave costs a whole wave).  Fewer, longer chunks mean fewer
// partial tiles to write and reduce but more truncating fp32 accumulations per TMEM block: measured on the layer1
// weight gradient of a 20-task step (1.17 M pixels), rel-L2 against the CUDA-core fp32 kernel / step time:
// 4 waves 5.5e-6 / 8.12 ms, 2 waves 1.1e-5 / 8.01 ms, 1 wave 2.3e-5 / 7.98 ms.  Two waves.  The CUDA-core kernel
// runs one CTA per (tap, chunk).
static int g_wgrad_waves = 2;   // full waves of (two CTAs per SM) per weight-gradient launch
int wgrad_chunks(long long M, int ntaps) {
  const int pairs = (ntaps + 1) / 2;
  long long want = (2LL * g_wgrad_waves * kNumSMs) / pairs;
  long long maxc = ceil_div(M, 64);
  if (want > maxc) want = maxc;
  return (int)(want < 1 ? 1 : want);
}
long long wgrad_pix_per_chunk(long long M, int chunks) { return ceil_div(ceil_div(M, chunks), 32) * 32; }

bool use_umma(int precision, int Cin, int Cout) {
  return precision != B200NP_PREC_FP32_SIMT && Cin == 64 && Cout == 64;
}

// bp0 / bp1: tensor-core images of the packed weights of source 0 / 1 (nullptr when absent)
int run_tapconv(const TapConvArgs& a, int precision, cudaStream_t st, const float* bp0 = nullptr, int ns0 = 0,
                const float* bp1 = nullptr, int ns1 = 0) {
  if (use_umma(precision, a.Cin, a.Cout)) {
    int rc = launch_tapconv_halo(a, bp0, ns0, bp1, ns1, precision, st);
    if (rc != B200NP_E_UNSUPPORTED) return rc;
    rc = launch_tapconv_umma(a, precision, st);
    if (rc != B200NP_E_UNSUPPORTED) return rc;
  }
  return launch_tapconv_simt(a, st);
}

}  // namespace

extern "C" size_t b200np_colsum_workspace(long long rows, int cols);
extern "C" int b200np_colsum(const float* x, float* out, long long rows, int cols, long long ld, void* ws,
                             size_t ws_bytes, void* stream);

extern "C" int b200np_pack_conv_weight(const float* w, float* wf, float* wd, int Cout, int Cin, int R,
                                       void* stream) {
  if (!w || (!wf && !wd) || Cout <= 0 || Cin <= 0 || R <= 0) return B200NP_E_BADARG;
  int total = Cout * Cin * R * R;
  pack_weight_kernel<<<(total + 255) / 256, 256, 0, as_stream(stream)>>>(w, wf, wd, Cout, Cin, R * R,
                                                                        Cout == 64 && Cin == 64);
  return launch_status();
}

extern "C" size_t b200np_packed_weight_floats(int Cout, int Cin, int R) {
  size_t base = (size_t)Cout * Cin * R * R;
  return (Cout == 64 && Cin == 64) ? 3 * base : base;
}

extern "C" int b200np_conv_fwd(const float* x, const float* wf, const float* bias, float* y, int N, int H, int W,
                               int Cin, int Cout, int R, int stride, const float* xs, const float* wsf,
                               const float* bias_s, int Cs, int stride_s, int act, int precision, uint32_t* relu_bits,
                               void* stream) {
  if (!x || !wf || !y || N <= 0 || H <= 0 || W <= 0) return B200NP_E_BADARG;
  if (relu_bits && !(use_umma(precision, Cin, Cout))) return B200NP_E_UNSUPPORTED;  // written by the tcgen05 epilogues only
  if ((R != 1 && R != 3) || (stride != 1 && stride != 2) || H % stride || W % stride) return B200NP_E_UNSUPPORTED;
  if (xs && (!wsf || Cs != Cin || stride_s < 1)) return B200NP_E_UNSUPPORTED;
  if (!aligned16(x) || !aligned16(wf) || !aligned16(y) || (xs && (!aligned16(xs) || !aligned16(wsf))))
    return B200NP_E_BADARG;
  TapConvArgs a{};
  a.src[0] = x; a.srcH[0] = H; a.srcW[0] = W; a.in_s[0] = stride; a.w[0] = wf;
  a.Cin = Cin; a.Cout = Cout; a.bias = bias; a.bias2 = xs ? bias_s : nullptr;
  a.dst = y; a.mask = nullptr; a.mask_bits = nullptr; a.relu_bits = relu_bits;
  a.N = N; a.OH = H / stride; a.OW = W / stride;
  a.dstH = a.OH; a.dstW = a.OW; a.dst_s = 1; a.dst_oy = 0; a.dst_ox = 0;
  a.act = act;
  int nt = 0;
  const int pad = R / 2;
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < R; ++s) a.taps[nt++] = Tap{0, (int8_t)(r - pad), (int8_t)(s - pad), (int8_t)(r * R + s)};
  if (xs) {
    a.src[1] = xs; a.srcH[1] = a.OH * stride_s; a.srcW[1] = a.OW * stride_s; a.in_s[1] = stride_s; a.w[1] = wsf;
    a.taps[nt++] = Tap{1, 0, 0, 0};
  }
  a.ntaps = nt;
  const bool img = Cin == 64 && Cout == 64;
  return run_tapconv(a, precision, as_stream(stream), img ? wf + (size_t)R * R * 4096 : nullptr, R * R,
                     (img && xs) ? wsf + 4096 : nullptr, 1);
}

extern "C" int b200np_conv_dgrad(const float* dy, const float* wd, float* dx, const float* mask_src,
                                 const uint32_t* mask_bits, int N, int H, int W, int Cin, int Cout, int R, int stride,
                                 const float* dys, const float* wsd, int Cs, int stride_s, int precision,
                                 void* stream) {
  if (!dy || !wd || !dx || N <= 0 || H <= 0 || W <= 0) return B200NP_E_BADARG;
  if ((R != 1 && R != 3) || (stride != 1 && stride != 2) || H % stride || W % stride) return B200NP_E_UNSUPPORTED;
  if (dys && (!wsd || Cs != Cout || stride_s != stride || stride != 2)) return B200NP_E_UNSUPPORTED;
  if (!aligned16(dy) || !aligned16(wd) || !aligned16(dx) || (mask_src && !aligned16(mask_src)) ||
      (dys && (!aligned16(dys) || !aligned16(wsd))))
    return B200NP_E_BADARG;
  const int pad = R / 2;
  const int OHc = H / stride, OWc = W / stride;  // dy geometry
  TapConvArgs a{};
  a.src[0] = dy; a.srcH[0] = OHc; a.srcW[0] = OWc; a.in_s[0] = 1; a.w[0] = wd;
  a.src[1] = dys; a.srcH[1] = OHc; a.srcW[1] = OWc; a.in_s[1] = 1; a.w[1] = wsd;
  a.Cin = Cout;  // reduction runs over the conv's output channels
  a.Cout = Cin;  // and produces the conv's input channels
  a.bias = a.bias2 = nullptr;
  if (mask_bits && Cin != 64) return B200NP_E_UNSUPPORTED;  // the packed gates are defined for 64-channel tensors
  a.dst = dx; a.mask = mask_src; a.mask_bits = mask_bits;
  a.N = N; a.dstH = H; a.dstW = W;
  a.act = B200NP_ACT_NONE;
  cudaStream_t st = as_stream(stream);
  const bool img = Cin == 64 && Cout == 64;
  if (stride == 1) {
    a.OH = H; a.OW = W; a.dst_s = 1; a.dst_oy = a.dst_ox = 0;
    int nt = 0;
    for (int r = 0; r < R; ++r)
      for (int s = 0; s < R; ++s) a.taps[nt++] = Tap{0, (int8_t)(pad - r), (int8_t)(pad - s), (int8_t)(r * R + s)};
    a.ntaps = nt;
    return run_tapconv(a, precision, st, img ? wd + (size_t)R * R * 4096 : nullptr, R * R);
  }
  // stride 2: one launch per parity class of the input pixel (iy,ix) = (2*oy+py, 2*ox+px).
  // y[o] = sum_r x[2o + r - pad] w[r]  =>  dx[i] = sum_{r : (i + pad - r) even} dy[(i + pad - r)/2] w[r]
  a.OH = OHc; a.OW = OWc; a.dst_s = 2;
  if (img && use_umma(precision, a.Cin, a.Cout)) {
    // all four classes from one staged dY halo (one launch, one accumulator set per class)
    TapConvArgs f = a;
    TapClasses cls{};
    cls.ncls = 4;
    int nt = 0;
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        const int c = py * 2 + px;
        cls.oy[c] = py; cls.ox[c] = px;
        for (int r = 0; r < R; ++r) {
          if ((py + pad - r) & 1) continue;
          for (int s = 0; s < R; ++s) {
            if ((px + pad - s) & 1) continue;
            cls.tap_cls[nt] = c;
            f.taps[nt++] = Tap{0, (int8_t)((py + pad - r) / 2), (int8_t)((px + pad - s) / 2), (int8_t)(r * R + s)};
          }
        }
        if (dys && c == 0) { cls.tap_cls[nt] = c; f.taps[nt++] = Tap{1, 0, 0, 0}; }
      }
    f.ntaps = nt;
    f.dst_oy = f.dst_ox = 0;
    if (R == 3) {
      int rc = launch_tapconv_halo(f, wd + (size_t)R * R * 4096, R * R, dys ? wsd + 4096 : nullptr, 1, precision, st, &cls);
      if (rc != B200NP_E_UNSUPPORTED) return rc;
    }
  }
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      int nt = 0;
      for (int r = 0; r < R; ++r) {
        if ((py + pad - r) & 1) continue;
        for (int s = 0; s < R; ++s) {
          if ((px + pad - s) & 1) continue;
          a.taps[nt++] = Tap{0, (int8_t)((py + pad - r) / 2), (int8_t)((px + pad - s) / 2), (int8_t)(r * R + s)};
        }
      }
      if (dys && py == 0 && px == 0) a.taps[nt++] = Tap{1, 0, 0, 0};
      a.ntaps = nt;
      a.dst_oy = py; a.dst_ox = px;
      int rc = run_tapconv(a, precision, st, img ? wd + (size_t)R * R * 4096 : nullptr, R * R,
                           (img && dys) ? wsd + 4096 : nullptr, 1);
      if (rc != B200NP_OK) return rc;
    }
  return B200NP_OK;
}

// Pixel chunks of the halo formulation of a 64->64 3x3 weight gradient (tapwgrad_halo.cu); 0 where it does not apply.
static int halo_chunks_for(int N, int OH, int OW, int Cin, int Cout, int R, int stride) {
  if (!(Cin == 64 && Cout == 64 && R == 3)) return 0;
  return stride == 1 ? tapwgrad_halo_chunks(N, OH, OW) : stride == 2 ? tapwgrad_halo_s2_chunks(N, OH, OW) : 0;
}

extern "C" size_t b200np_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int R, int stride) {
  if (N <= 0 || stride <= 0) return 0;
  long long M = (long long)N * (H / stride) * (W / stride);
  int nt = R * R + 1;  // room for a fused skip-projection tap
  int chunks = wgrad_chunks(M, nt);
  const int hc = halo_chunks_for(N, H / stride, W / stride, Cin, Cout, R, stride);
  if (hc > chunks) chunks = hc;
  size_t part = (size_t)chunks * nt * Cout * Cin * sizeof(float);
  size_t dbw = b200np_colsum_workspace(M, Cout), dbp = (size_t)chunks * Cout * sizeof(float);
  return part + (dbw > dbp ? dbw : dbp);
}

extern "C" int b200np_conv_wgrad(const float* x, const float* dy, float* dw, float* db, int N, int H, int W, int Cin,
                                 int Cout, int R, int stride, const float* xs, float* dws, int stride_s,
                                 int precision, void* ws, size_t ws_bytes, void* stream) {
  if (!x || !dy || !dw || N <= 0 || H <= 0 || W <= 0) return B200NP_E_BADARG;
  if (xs && (!dws || Cin != 64 || Cout != 64 || stride_s < 1 || !aligned16(xs))) return B200NP_E_UNSUPPORTED;
  if ((R != 1 && R != 3) || (stride != 1 && stride != 2) || H % stride || W % stride) return B200NP_E_UNSUPPORTED;
  if (!aligned16(x) || !aligned16(dy) || !aligned16(ws)) return B200NP_E_BADARG;
  if (!ws || ws_bytes < b200np_conv_wgrad_workspace(N, H, W, Cin, Cout, R, stride)) return B200NP_E_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  TapWgradArgs a{};
  a.src = x; a.srcH = H; a.srcW = W; a.in_s = stride; a.Cin = Cin;
  a.dy = dy; a.N = N; a.OH = H / stride; a.OW = W / stride; a.Cout = Cout;
  const int pad = R / 2;
  int nt = 0;
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < R; ++s) a.taps[nt++] = Tap{0, (int8_t)(r - pad), (int8_t)(s - pad), (int8_t)(r * R + s)};
  if (xs) {  // the skip projection sees the same dy: one more tap on a second source
    a.src2 = xs; a.src2H = a.OH * stride_s; a.src2W = a.OW * stride_s; a.in_s2 = stride_s;
    a.taps[nt++] = Tap{1, 0, 0, (int8_t)(R * R)};
  }
  a.ntaps = nt;
  const long long M = (long long)N * a.OH * a.OW;
  a.chunks = wgrad_chunks(M, nt);
  a.pix_per_chunk = wgrad_pix_per_chunk(M, a.chunks);
  a.part = (float*)ws;
  const int per = nt * Cout * Cin;
  size_t part_bytes = (size_t)a.chunks * per * sizeof(float);
  int rc = B200NP_E_UNSUPPORTED;
  bool db_fused = false;
  if (use_umma(precision, Cin, Cout)) {
    const int hc = halo_chunks_for(N, a.OH, a.OW, Cin, Cout, R, stride);
    if (hc > 0) {   // tile-staged taps (tapwgrad_halo.cu); sets a.chunks = hc
      const size_t pb = (size_t)hc * per * sizeof(float);
      a.part_db = db ? (float*)((char*)ws + pb) : nullptr;
      rc = launch_tapwgrad_halo(a, precision, st);
      if (rc == B200NP_OK) part_bytes = pb;
      else if (rc == B200NP_E_UNSUPPORTED) a.chunks = wgrad_chunks(M, nt);
    }
    if (rc == B200NP_E_UNSUPPORTED) {
      a.part_db = db ? (float*)((char*)ws + part_bytes) : nullptr;   // bias gradient from the dy tiles the kernel stages
      rc = launch_tapwgrad_umma(a, precision, st);
    }
    db_fused = rc == B200NP_OK && db;
  }
  if (rc == B200NP_E_UNSUPPORTED) {
    a.part_db = nullptr;
    rc = launch_tapwgrad_simt(a, st);
  }
  if (rc != B200NP_OK) return rc;
  rc = launch_reduce_partials(a.part, dw, a.chunks, per, ReduceMap{1, R * R, Cout, Cin, dws}, st);
  if (rc != B200NP_OK) return rc;
  if (db_fused) return launch_reduce_partials(a.part_db, db, a.chunks, Cout, ReduceMap{0, 0, 0, 0, nullptr}, st);
  if (db) {
    rc = b200np_colsum(dy, db, M, Cout, Cout, (char*)ws + part_bytes, ws_bytes - part_bytes, stream);
    if (rc != B200NP_OK) return rc;
  }
  return B200NP_OK;
}

// diagnostics (tools/run_dominant_kernel.py, bench.py): pixel chunks per weight-gradient launch, in full waves
extern "C" void b200np_debug_set_wgrad_waves(int w) { g_wgrad_waves = w < 1 ? 1 : w; }
