// Elementwise / reduction kernels: HBM-bound, coalesced, vectorised where alignment allows.
#include <float.h>
#include <math.h>

#include "common.cuh"

using namespace b200np;

extern "C" const char* b200np_strerror(int code) {
  switch (code) {
    case B200NP_OK: return "ok";
    case B200NP_E_BADARG: return "bad argument (dimension / pointer / alignment precondition)";
    case B200NP_E_LAUNCH: return "CUDA launch failure";
    case B200NP_E_WORKSPACE: return "workspace too small";
    case B200NP_E_UNSUPPORTED: return "unsupported configuration";
    default: return "unknown error";
  }
}
namespace b200np { std::atomic<long long> g_launches{0}; }
extern "C" int b200np_version(void) { return B200NP_VERSION; }
extern "C" long long b200np_launch_count(void) { return b200np::g_launches.load(); }
extern "C" int b200np_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return B200NP_E_LAUNCH;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
    return B200NP_E_LAUNCH;
  return major == 10 ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
__global__ void fill_kernel(float* __restrict__ x, long long n, float v) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += st) x[i] = v;
}
extern "C" int b200np_fill(float* x, long long n, float value, void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!x) return B200NP_E_BADARG;
  fill_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(x, n, value);
  return launch_status();
}

__global__ void axpy_kernel(float* __restrict__ y, const float* __restrict__ x, long long n, float a) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += st) y[i] = fmaf(a, x[i], y[i]);
}
extern "C" int b200np_axpy(float* y, const float* x, long long n, float a, void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!x || !y) return B200NP_E_BADARG;
  axpy_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(y, x, n, a);
  return launch_status();
}

// Segment i of a launch is dst[off_i .. off_i + n_i) and src_i, up to 64 segments per launch, passed by value.
// kAdd false (copy): dst = src_i, or 0 where src_i is NULL.  kAdd true (accumulate): dst += src_i, and a NULL src_i
// leaves its range alone; float4 where both sides are 16-byte aligned (always so for FlatParams views), then a scalar
// tail.  Plain fp32 adds, one per element: deterministic.
constexpr int kSegsPerLaunch = 64;
struct CopySegs {
  const float* src[kSegsPerLaunch];
  long long off[kSegsPerLaunch];
  long long n[kSegsPerLaunch];
};
template <bool kAdd>
__device__ __forceinline__ void multi_segment(const float* __restrict__ s, float* __restrict__ d, const long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long st = (long long)gridDim.x * blockDim.x;
  // __ldg: once this body is inlined, restrict alone no longer gives the read-only loads the copy kernel always had
  if (!kAdd) {
    if (s) for (; i < n; i += st) d[i] = __ldg(s + i);
    else for (; i < n; i += st) d[i] = 0.f;
    return;
  }
  if (!s) return;
  if (((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
    const long long n4 = n >> 2;
    const float4* __restrict__ s4 = reinterpret_cast<const float4*>(s);
    float4* __restrict__ d4 = reinterpret_cast<float4*>(d);
    for (long long q = i; q < n4; q += st) {
      const float4 a = __ldg(s4 + q);
      float4 b = d4[q];
      b.x += a.x, b.y += a.y, b.z += a.z, b.w += a.w;
      d4[q] = b;
    }
    i += n4 << 2;
  }
  for (; i < n; i += st) d[i] += __ldg(s + i);
}
// two kernels rather than one template, so that profiles and the kernel-route tests name each by its own name
__global__ void multi_copy_kernel(const CopySegs g, float* __restrict__ dst) {
  multi_segment<false>(g.src[blockIdx.y], dst + g.off[blockIdx.y], g.n[blockIdx.y]);
}
__global__ void multi_accumulate_kernel(const CopySegs g, float* __restrict__ dst) {
  multi_segment<true>(g.src[blockIdx.y], dst + g.off[blockIdx.y], g.n[blockIdx.y]);
}

template <bool kAdd>
static int multi_segments(const float* const* src, const long long* dst_off, const long long* numel, int nseg,
                          float* dst, void* stream) {
  if (nseg <= 0) return B200NP_OK;
  if (!src || !dst_off || !numel || !dst) return B200NP_E_BADARG;
  for (int base = 0; base < nseg; base += kSegsPerLaunch) {
    CopySegs g{};
    const int cnt = nseg - base < kSegsPerLaunch ? nseg - base : kSegsPerLaunch;
    long long mx = 1;
    for (int i = 0; i < cnt; ++i) {
      if (numel[base + i] < 0 || dst_off[base + i] < 0) return B200NP_E_BADARG;
      g.src[i] = src[base + i]; g.off[i] = dst_off[base + i]; g.n[i] = numel[base + i];
      if (g.n[i] > mx) mx = g.n[i];
    }
    long long bx = (mx + 1023) / 1024;   // 256 threads x 4 elements
    if (bx > 64) bx = 64;
    (kAdd ? multi_accumulate_kernel : multi_copy_kernel)<<<dim3((unsigned)bx, (unsigned)cnt), 256, 0,
                                                            as_stream(stream)>>>(g, dst);
    int rc = launch_status();
    if (rc != B200NP_OK) return rc;
  }
  return B200NP_OK;
}
extern "C" int b200np_multi_copy(const float* const* src, const long long* dst_off, const long long* numel, int nseg,
                                 float* dst, void* stream) {
  return multi_segments<false>(src, dst_off, numel, nseg, dst, stream);
}
extern "C" int b200np_multi_accumulate(const float* const* src, const long long* dst_off, const long long* numel,
                                       int nseg, float* dst, void* stream) {
  return multi_segments<true>(src, dst_off, numel, nseg, dst, stream);
}

// ------------------------------------------------------------------------------------------------
// Device-side task assembly (dataset/shapenet_distractor.py:233-234,256-259; utils/utils.py:26-30):
// out[m, c, y, x] = float(255 - bank[rows[m], y, x, c]) / 255   -- uint8 image bank resident in HBM, channel-last,
// gathered by row index into the fp32 NCHW batch the model consumes.  HBM-bound byte work: 1 B read, 4 B written
// per element; a thread converts 4 consecutive pixels of one channel plane (uchar4 -> float4 when C == 1).
// ------------------------------------------------------------------------------------------------
__global__ void gather_images_u8_kernel(const uint8_t* __restrict__ bank, const int32_t* __restrict__ rows,
                                        float* __restrict__ out, long long M, int H, int W, int C) {
  const long long plane = (long long)H * W, per = plane * C;
  const long long quads = M * per / 4;
  long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long st = (long long)gridDim.x * blockDim.x;
  for (; q < quads; q += st) {
    const long long e = q * 4;                       // first output element of this quad
    const long long m = e / per, r = e - m * per;
    const int c = (int)(r / plane);
    const long long pix = r - (long long)c * plane;  // plane % 4 == 0: the quad stays inside one channel plane
    const uint8_t* src = bank + (long long)__ldg(rows + m) * per + pix * C + c;
    float4 v;
    if (C == 1) {
      const uchar4 u = __ldg(reinterpret_cast<const uchar4*>(src));
      v = make_float4((float)(255 - u.x) / 255.0f, (float)(255 - u.y) / 255.0f, (float)(255 - u.z) / 255.0f,
                      (float)(255 - u.w) / 255.0f);
    } else {
      v = make_float4((float)(255 - __ldg(src)) / 255.0f, (float)(255 - __ldg(src + C)) / 255.0f,
                      (float)(255 - __ldg(src + 2 * C)) / 255.0f, (float)(255 - __ldg(src + 3 * C)) / 255.0f);
    }
    *reinterpret_cast<float4*>(out + e) = v;
  }
}
extern "C" int b200np_gather_images_u8(const uint8_t* bank, const int32_t* rows, float* out, long long M, int H, int W,
                                       int C, void* stream) {
  if (M <= 0) return B200NP_OK;
  if (!bank || !rows || !out || H <= 0 || W <= 0 || C <= 0) return B200NP_E_BADARG;
  if (((long long)H * W) % 4 != 0 || !aligned16(out) || (reinterpret_cast<uintptr_t>(bank) & 3u)) return B200NP_E_UNSUPPORTED;
  const long long quads = M * H * W * C / 4;
  gather_images_u8_kernel<<<ew_grid(quads, 256), 256, 0, as_stream(stream)>>>(bank, rows, out, M, H, W, C);
  return launch_status();
}

__global__ void act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                               float* __restrict__ dz, long long n, int act) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += st) {
    float g = dy[i], o = y[i];
    dz[i] = act == B200NP_ACT_RELU ? (o > 0.f ? g : 0.f) : act == B200NP_ACT_TANH ? g * (1.f - o * o) : g;
  }
}
extern "C" int b200np_act_bwd(const float* dy, const float* y, float* dz, long long n, int act,
                              void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!dy || !y || !dz) return B200NP_E_BADARG;
  act_bwd_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(dy, y, dz, n, act);
  return launch_status();
}

__global__ void scale_dev_kernel(const float* __restrict__ x, const float* __restrict__ s,
                                 float* __restrict__ y, long long n) {
  float a = __ldg(s);
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += st) y[i] = a * x[i];
}
extern "C" int b200np_scale_by_device_scalar(const float* x, const float* scale, float* y, long long n,
                                             void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!x || !scale || !y) return B200NP_E_BADARG;
  scale_dev_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(x, scale, y, n);
  return launch_status();
}

__global__ void repeat_rows_kernel(const float* __restrict__ x, float* __restrict__ y, long long rows_in,
                                   int rep, int cols) {
  long long total = rows_in * rep * cols;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < total; i += st) {
    long long r = i / cols;
    int c = (int)(i - r * cols);
    y[i] = x[(r / rep) * cols + c];
  }
}
extern "C" int b200np_repeat_rows(const float* x, float* y, long long rows_in, int rep, int cols,
                                  void* stream) {
  long long n = rows_in * rep * cols;
  if (n <= 0) return B200NP_OK;
  if (!x || !y) return B200NP_E_BADARG;
  repeat_rows_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(x, y, rows_in, rep, cols);
  return launch_status();
}
__global__ void repeat_rows_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx,
                                       long long rows_in, int rep, int cols) {
  long long total = rows_in * cols;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < total; i += st) {
    long long r = i / cols;
    int c = (int)(i - r * cols);
    float s = 0.f;
    for (int k = 0; k < rep; ++k) s += dy[(r * rep + k) * cols + c];
    dx[i] = s;
  }
}
extern "C" int b200np_repeat_rows_bwd(const float* dy, float* dx, long long rows_in, int rep, int cols,
                                      void* stream) {
  long long n = rows_in * cols;
  if (n <= 0) return B200NP_OK;
  if (!dy || !dx) return B200NP_E_BADARG;
  repeat_rows_bwd_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(dy, dx, rows_in, rep, cols);
  return launch_status();
}

// out = alpha * a * b * c (b, c nullable = 1): the elementwise products of the second-order terms (tanh'' = -2 y dy v,
// the MSE loss's constant Hessian 2/R)
__global__ void mul3_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                            float alpha, float* __restrict__ out, long long n) {
  const long long st = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += st)
    out[i] = alpha * a[i] * (b ? b[i] : 1.f) * (c ? c[i] : 1.f);
}
extern "C" int b200np_mul3(const float* a, const float* b, const float* c, float alpha, float* out, long long n,
                           void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!a || !out) return B200NP_E_BADARG;
  mul3_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(a, b, c, alpha, out, n);
  return launch_status();
}

// ------------------------------------------------------------------------------------------------
// Partial-sum reducer shared by the split-K weight gradients and the column sums.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ part, float* __restrict__ out,
                                                              int nparts, int n, b200np::ReduceMap map) {
  __shared__ float sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  float s = 0.f;
  if (j < n) {
#pragma unroll 4
    for (int p = ty; p < nparts; p += 8) s += part[(long long)p * n + j];
  }
  sm[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && j < n) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sm[k][tx];
    if (map.kind == 0) {
      out[j] = t;
    } else if (map.kind == 1) {
      const int ci = j % map.c, r = j / map.c;
      const int co = r % map.b, tp = r / map.b;
      if (tp < map.a) out[((long long)co * map.c + ci) * map.a + tp] = t;
      else map.out2[(long long)co * map.c + ci] = t;   // fused 1x1 skip projection: [Cout][Cin]
    } else {
      const int co = j / map.b, k = j - co * map.b;
      if (k < map.a) out[co * map.a + k] = t;
      else if (k == map.a && map.out2) map.out2[co] = t;
    }
  }
}
__device__ __forceinline__ void reduce_store(float* __restrict__ out, int j, float t, const b200np::ReduceMap& map) {
  if (map.kind == 0) {
    out[j] = t;
  } else if (map.kind == 1) {
    const int ci = j % map.c, r = j / map.c;
    const int co = r % map.b, tp = r / map.b;
    if (tp < map.a) out[((long long)co * map.c + ci) * map.a + tp] = t;
    else map.out2[(long long)co * map.c + ci] = t;
  } else {
    const int co = j / map.b, k = j - co * map.b;
    if (k < map.a) out[co * map.a + k] = t;
    else if (k == map.a && map.out2) map.out2[co] = t;
  }
}
// Four columns per thread (16-byte loads, 512 contiguous bytes per warp instruction) and LANES partial-lanes per column
// group: lane ty sums partials ty, ty + LANES, ... in order, then the lanes are folded 0..LANES-1 -- a fixed order, so the
// result is deterministic.  The partials were written a moment ago and sit in L2; these reducers are serialised between
// the weight-gradient kernels at the end of the step, so what counts is bytes in flight per SM: n / 128 blocks is only
// ~2 per SM, hence 32 lanes (1024 threads) once there are enough partials.
template <int LANES>
__global__ void __launch_bounds__(32 * LANES) reduce_partials_vec4_kernel(const float* __restrict__ part,
                                                                           float* __restrict__ out, int nparts, int n,
                                                                           b200np::ReduceMap map) {
  __shared__ float4 sm[LANES][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = (blockIdx.x * 32 + tx) * 4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (j < n) {
#pragma unroll 4
    for (int p = ty; p < nparts; p += LANES) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(part + (long long)p * n + j));
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  }
  sm[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && j < n) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < LANES; ++k) {
      const float4 v = sm[k][tx];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    reduce_store(out, j, t.x, map);
    reduce_store(out, j + 1, t.y, map);
    reduce_store(out, j + 2, t.z, map);
    reduce_store(out, j + 3, t.w, map);
  }
}
namespace b200np {
int launch_reduce_partials(const float* part, float* out, int nparts, int n, ReduceMap map, cudaStream_t st) {
  if (n <= 0) return B200NP_OK;
  if ((n & 3) == 0 && aligned16(part) && nparts >= 128)
    reduce_partials_vec4_kernel<32><<<(n / 4 + 31) / 32, 1024, 0, st>>>(part, out, nparts, n, map);
  else if ((n & 3) == 0 && aligned16(part) && nparts >= 16)
    reduce_partials_vec4_kernel<8><<<(n / 4 + 31) / 32, 256, 0, st>>>(part, out, nparts, n, map);
  else
    reduce_partials_kernel<<<(n + 31) / 32, 256, 0, st>>>(part, out, nparts, n, map);
  return launch_status();
}
}  // namespace b200np

// ------------------------------------------------------------------------------------------------
// Column sums (bias gradients), deterministic two-stage: blocks of (32 columns x 8 row lanes)
// reduce a contiguous row chunk into ws[chunk][col]; a second kernel folds the chunks in order.
// ------------------------------------------------------------------------------------------------
constexpr int kColsumChunksMax = 592;  // 4 x 148
static int colsum_chunks(long long rows) {
  long long c = ceil_div(rows, 256);
  if (c > kColsumChunksMax) c = kColsumChunksMax;
  return (int)(c < 1 ? 1 : c);
}
__global__ void colsum_stage1(const float* __restrict__ x, float* __restrict__ part, long long rows,
                              int cols, long long ld, int chunks) {
  __shared__ float sm[8][33];
  int c = blockIdx.x * 32 + threadIdx.x;
  int chunk = blockIdx.y;
  long long per = (rows + chunks - 1) / chunks;
  long long r0 = chunk * per, r1 = r0 + per < rows ? r0 + per : rows;
  float s = 0.f;
  if (c < cols)
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) s += x[r * ld + c];
  sm[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sm[k][threadIdx.x];
    part[(long long)chunk * cols + c] = t;
  }
}
extern "C" size_t b200np_colsum_workspace(long long rows, int cols) {
  return (size_t)colsum_chunks(rows) * (size_t)cols * sizeof(float);
}
extern "C" int b200np_colsum(const float* x, float* out, long long rows, int cols, long long ld, void* ws,
                             size_t ws_bytes, void* stream) {
  if (cols <= 0) return B200NP_OK;
  if (!x || !out || rows < 0 || ld < cols) return B200NP_E_BADARG;
  if (rows == 0) return b200np_fill(out, cols, 0.f, stream);
  int chunks = colsum_chunks(rows);
  if (!ws || ws_bytes < (size_t)chunks * cols * sizeof(float)) return B200NP_E_WORKSPACE;
  dim3 grid((cols + 31) / 32, chunks), block(32, 8);
  colsum_stage1<<<grid, block, 0, as_stream(stream)>>>(x, (float*)ws, rows, cols, ld, chunks);
  int rc = launch_reduce_partials((const float*)ws, out, chunks, cols, ReduceMap{0, 0, 0, 0, nullptr}, as_stream(stream));
  if (rc != B200NP_OK) return rc;
  return launch_status(1);
}

// ------------------------------------------------------------------------------------------------
__global__ void max_reduce_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  __shared__ float red[32];
  float m = -INFINITY;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, x[i]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
    t = warp_max(t);
    if (threadIdx.x == 0) out[0] = t;
  }
}
extern "C" int b200np_max_reduce(const float* x, long long n, float* out, void* stream) {
  if (!x || !out || n <= 0) return B200NP_E_BADARG;
  max_reduce_kernel<<<1, 1024, 0, as_stream(stream)>>>(x, n, out);
  return launch_status();
}

// ------------------------------------------------------------------------------------------------
// CNP context aggregation: feats [T,nc,D] -> out [T,D]; one thread per (task, feature), the
// context loop strides by D so every load is coalesced across the warp.
// ------------------------------------------------------------------------------------------------
__global__ void ctx_agg_fwd_kernel(const float* __restrict__ f, float* __restrict__ out,
                                   int32_t* __restrict__ idx, int T, int nc, int D, int mode) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * D) return;
  int t = (int)(i / D), c = (int)(i - (long long)t * D);
  const float* p = f + (long long)t * nc * D + c;
  if (mode == 0) {
    float s = 0.f;
    for (int j = 0; j < nc; ++j) s += p[(long long)j * D];
    out[i] = s / (float)nc;
  } else {
    float m = p[0];
    int a = 0;
    for (int j = 1; j < nc; ++j) {
      float v = p[(long long)j * D];
      if (v > m) { m = v; a = j; }  // strict '>' keeps the FIRST maximum (torch.max(dim) rule)
    }
    out[i] = m;
    if (idx) idx[i] = a;
  }
}
// D % 4 == 0, 16-byte aligned: thread = four consecutive features of one task; the context loop issues four
// independent 16-byte loads per trip (a warp instruction covers 512 contiguous bytes), results leave as one float4 /
// int4.  Same element order and comparison rule as the scalar kernel, so the results are bit-identical.
__global__ void __launch_bounds__(128) ctx_agg_fwd_vec4_kernel(const float* __restrict__ f, float* __restrict__ out,
                                                               int32_t* __restrict__ idx, int T, int nc, int D4,
                                                               int mode) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * D4) return;
  const int t = (int)(i / D4), c4 = (int)(i - (long long)t * D4);
  const float4* p = reinterpret_cast<const float4*>(f) + (long long)t * nc * D4 + c4;
  if (mode == 0) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = 0;
    for (; j + 4 <= nc; j += 4) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(p + (long long)(j + u) * D4);
#pragma unroll
      for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; j < nc; ++j) {
      const float4 v = __ldg(p + (long long)j * D4);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const float inv = (float)nc;
    reinterpret_cast<float4*>(out)[i] = make_float4(s.x / inv, s.y / inv, s.z / inv, s.w / inv);
  } else {
    float4 m = __ldg(p);
    int4 a = make_int4(0, 0, 0, 0);
    int j = 1;
    for (; j + 4 <= nc; j += 4) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(p + (long long)(j + u) * D4);
#pragma unroll
      for (int u = 0; u < 4; ++u) {   // strict '>' keeps the FIRST maximum (torch.max(dim) rule)
        if (v[u].x > m.x) { m.x = v[u].x; a.x = j + u; }
        if (v[u].y > m.y) { m.y = v[u].y; a.y = j + u; }
        if (v[u].z > m.z) { m.z = v[u].z; a.z = j + u; }
        if (v[u].w > m.w) { m.w = v[u].w; a.w = j + u; }
      }
    }
    for (; j < nc; ++j) {
      const float4 v = __ldg(p + (long long)j * D4);
      if (v.x > m.x) { m.x = v.x; a.x = j; }
      if (v.y > m.y) { m.y = v.y; a.y = j; }
      if (v.z > m.z) { m.z = v.z; a.z = j; }
      if (v.w > m.w) { m.w = v.w; a.w = j; }
    }
    reinterpret_cast<float4*>(out)[i] = m;
    if (idx) reinterpret_cast<int4*>(idx)[i] = a;
  }
}
__global__ void ctx_agg_bwd_kernel(const float* __restrict__ dout, const int32_t* __restrict__ idx,
                                   float* __restrict__ df, int T, int nc, int D, int mode) {
  long long n = (long long)T * nc * D;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, st = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += st) {
    int c = (int)(i % D);
    long long tj = i / D;
    int j = (int)(tj % nc);
    long long t = tj / nc;
    float g = dout[t * D + c];
    df[i] = mode == 0 ? g / (float)nc : (idx[t * D + c] == j ? g : 0.f);
  }
}
extern "C" int b200np_ctx_aggregate_fwd(const float* feats, float* out, int32_t* idx, int T, int nc, int D,
                                        int mode, void* stream) {
  if (!feats || !out || T <= 0 || nc <= 0 || D <= 0 || (mode != 0 && mode != 1)) return B200NP_E_BADARG;
  if (mode == 1 && !idx) return B200NP_E_BADARG;
  long long n = (long long)T * D;
  if (D % 4 == 0 && aligned16(feats) && aligned16(out) && (!idx || aligned16(idx))) {
    ctx_agg_fwd_vec4_kernel<<<(unsigned)ceil_div(n / 4, 128), 128, 0, as_stream(stream)>>>(feats, out, idx, T, nc, D / 4, mode);
    return launch_status();
  }
  ctx_agg_fwd_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, as_stream(stream)>>>(feats, out, idx, T, nc, D, mode);
  return launch_status();
}
extern "C" int b200np_ctx_aggregate_bwd(const float* dout, const int32_t* idx, float* dfeats, int T, int nc,
                                        int D, int mode, void* stream) {
  if (!dout || !dfeats || T <= 0 || nc <= 0 || D <= 0 || (mode != 0 && mode != 1)) return B200NP_E_BADARG;
  if (mode == 1 && !idx) return B200NP_E_BADARG;
  long long n = (long long)T * nc * D;
  ctx_agg_bwd_kernel<<<ew_grid(n, 256), 256, 0, as_stream(stream)>>>(dout, idx, dfeats, T, nc, D, mode);
  return launch_status();
}

// ------------------------------------------------------------------------------------------------
// Bayesian context aggregation (networks/CNPDistractor.py:60-75,104-110): per task and feature, with
//   var_i = 1e-5 + softplus(s_i),  a_i = 1 / var_i,  sigma_z = 1 / (1 + sum_i a_i),  r = sigma_z * sum_i a_i mu_i
// (prior mean 0, variance 1).  softplus follows torch (threshold 20).  One thread per (task, feature).
// Backward:  d mu_i = dr * sigma_z * a_i,   d s_i = -dr * sigma_z * (mu_i - r) * a_i^2 * sigmoid(s_i).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_t(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__global__ void baco_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ s, float* __restrict__ r,
                                int T, int nc, int D) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * D) return;
  const int t = (int)(i / D), dd = (int)(i - (long long)t * D);
  float A = 0.f, B = 0.f;
  for (int j = 0; j < nc; ++j) {
    const long long o = ((long long)t * nc + j) * D + dd;
    const float a = 1.f / (1e-5f + softplus_t(s[o]));
    A += a;
    B = fmaf(a, mu[o], B);
  }
  r[i] = B / (1.f + A);
}
__global__ void baco_bwd_kernel(const float* __restrict__ dr, const float* __restrict__ mu, const float* __restrict__ s,
                                const float* __restrict__ r, float* __restrict__ dmu, float* __restrict__ ds, int T,
                                int nc, int D) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * D) return;
  const int t = (int)(i / D), dd = (int)(i - (long long)t * D);
  float A = 0.f;
  for (int j = 0; j < nc; ++j) A += 1.f / (1e-5f + softplus_t(s[((long long)t * nc + j) * D + dd]));
  const float sz = 1.f / (1.f + A), g = dr[i] * sz, ri = r[i];
  for (int j = 0; j < nc; ++j) {
    const long long o = ((long long)t * nc + j) * D + dd;
    const float x = s[o], a = 1.f / (1e-5f + softplus_t(x));
    const float sig = x > 20.f ? 1.f : 1.f / (1.f + expf(-x));
    dmu[o] = g * a;
    ds[o] = -g * (mu[o] - ri) * a * a * sig;
  }
}
extern "C" int b200np_baco_fwd(const float* mu, const float* s, float* r, int T, int nc, int D, void* stream) {
  if (!mu || !s || !r || T <= 0 || nc <= 0 || D <= 0) return B200NP_E_BADARG;
  const long long n = (long long)T * D;
  baco_fwd_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, as_stream(stream)>>>(mu, s, r, T, nc, D);
  return launch_status();
}
extern "C" int b200np_baco_bwd(const float* dr, const float* mu, const float* s, const float* r, float* dmu, float* ds,
                               int T, int nc, int D, void* stream) {
  if (!dr || !mu || !s || !r || !dmu || !ds || T <= 0 || nc <= 0 || D <= 0) return B200NP_E_BADARG;
  const long long n = (long long)T * D;
  baco_bwd_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, as_stream(stream)>>>(dr, mu, s, r, dmu, ds, T, nc, D);
  return launch_status();
}

// ------------------------------------------------------------------------------------------------
// Losses: one block; rows are tiny ([T*nt, 2|4]).  Writes the mean loss and d loss / d mu.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sgn(float v) { return (v > 0.f) - (v < 0.f); }

// One row of the loss: returns its term of the sum, writes d mu of the row (already divided by R).
__device__ __forceinline__ float loss_row(const float* __restrict__ m, const float* __restrict__ t, float* __restrict__ d,
                                          int L, int kind, float invR) {
  if (kind == 0) {  // trainer/losses.py:35-36
    const float2 mm = *reinterpret_cast<const float2*>(m);
    float e0 = t[0] - mm.x, e1 = t[1] - mm.y;
    float nrm = sqrtf(e0 * e0 + e1 * e1);
    if (d) *reinterpret_cast<float2*>(d) = make_float2(-e0 / nrm * invR, -e1 / nrm * invR);
    return nrm;
  } else if (kind == 1) {  // trainer/losses.py:50-57
    float q[4], g[4], nrm = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) nrm += m[k] * m[k];
    nrm = sqrtf(nrm);
    float pos = 0.f, neg = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      q[k] = m[k] / nrm;
      pos += fabsf(t[k] - q[k]);
      neg += fabsf(-t[k] - q[k]);
    }
    if (d) {
      float wp = pos < neg ? 1.f : (pos > neg ? 0.f : 0.5f);  // torch.minimum splits ties evenly
      float dot = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        g[k] = -(wp * sgn(t[k] - q[k]) + (1.f - wp) * sgn(-t[k] - q[k]));
        dot += g[k] * q[k];
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) d[k] = (g[k] - q[k] * dot) / nrm * invR;
    }
    return fminf(pos, neg);
  } else if (kind == 2) {  // trainer/losses.py:59-61
    const float2 mm = *reinterpret_cast<const float2*>(m);
    float e0 = t[0] - mm.x, e1 = t[1] - mm.y;
    if (d) *reinterpret_cast<float2*>(d) = make_float2(-2.f * e0 * invR, -2.f * e1 * invR);
    return e0 * e0 + e1 * e1;
  }
  // degree error, trainer/losses.py:63-76 (evaluation only)
  const float r2d = 180.f / 3.14159265358979323846f;
  float gt = t[L - 1] * r2d;
  float a = acosf(m[0]);
  if (m[1] < 0.f) a = -a + 2.f * 3.14159265358979323846f;
  a *= r2d;
  return fminf(fabsf(gt - a), fminf(fabsf(gt + 360.f - a), fabsf(gt - (a + 360.f))));
}

// The hot path's losses have a few hundred rows (T * nt): ONE block, one launch, deterministic block reduction.
__global__ void loss_kernel(const float* __restrict__ mu, const float* __restrict__ y, float* __restrict__ loss,
                            float* __restrict__ dmu, long long R, int out, int L, int kind) {
  __shared__ float red[32];
  float acc = 0.f;
  const float invR = 1.f / (float)R;
  for (long long r = threadIdx.x; r < R; r += blockDim.x)
    acc += loss_row(mu + r * out, y + r * L, dmu ? dmu + r * out : nullptr, L, kind, invR);
  float tot = block_sum(acc, red);
  if (threadIdx.x == 0) loss[0] = tot * invR;
}
// Large row counts (evaluation over whole datasets, the HBM-bandwidth measurement of bench.py): grid-stride over rows,
// per-block partial sums, and the LAST block to finish (atomic ticket) adds the partials in block order -- one launch,
// deterministic.  The partial buffer and the ticket are library globals: two such launches must not overlap (the
// single-block kernel above, which the training step uses, has no shared state).
constexpr int kLossBlocks = 4 * kNumSMs;
__device__ float g_loss_part[kLossBlocks];
__device__ unsigned int g_loss_ticket = 0;
__device__ __forceinline__ void loss_finish(float acc, float* red, bool* last, float* __restrict__ loss, float invR) {
  float tot = block_sum(acc, red);
  if (threadIdx.x == 0) {
    g_loss_part[blockIdx.x] = tot;
    __threadfence();
    *last = atomicAdd(&g_loss_ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!*last) return;
  __threadfence();
  float s = 0.f;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) s += __ldcg(g_loss_part + b);
  s = block_sum(s, red);
  if (threadIdx.x == 0) { loss[0] = s * invR; g_loss_ticket = 0; }
}
__global__ void __launch_bounds__(256) loss_multi_kernel(const float* __restrict__ mu, const float* __restrict__ y,
                                                         float* __restrict__ loss, float* __restrict__ dmu, long long R,
                                                         int out, int L, int kind) {
  __shared__ float red[32];
  __shared__ bool last;
  float acc = 0.f;
  const float invR = 1.f / (float)R;
  const long long st = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += st)
    acc += loss_row(mu + r * out, y + r * L, dmu ? dmu + r * out : nullptr, L, kind, invR);
  loss_finish(acc, red, &last, loss, invR);
}
// Two-wide rows with two-wide labels (distractor / azimuth with L = 2): a thread takes TWO consecutive rows, so every
// access is 16 bytes and a warp instruction covers 512 contiguous bytes (the scalar-row form reaches 64 % of the HBM peak).
__global__ void __launch_bounds__(256) loss_multi_vec_kernel(const float* __restrict__ mu, const float* __restrict__ y,
                                                             float* __restrict__ loss, float* __restrict__ dmu, long long R,
                                                             int kind) {
  __shared__ float red[32];
  __shared__ bool last;
  float acc = 0.f;
  const float invR = 1.f / (float)R;
  const long long st = (long long)gridDim.x * blockDim.x, pairs = R >> 1;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < pairs; q += st) {
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu) + q), t = __ldg(reinterpret_cast<const float4*>(y) + q);
    const float a0 = t.x - m.x, a1 = t.y - m.y, b0 = t.z - m.z, b1 = t.w - m.w;
    float4 d;
    if (kind == 0) {
      const float na = sqrtf(a0 * a0 + a1 * a1), nb = sqrtf(b0 * b0 + b1 * b1);
      acc += na + nb;
      d = make_float4(-a0 / na * invR, -a1 / na * invR, -b0 / nb * invR, -b1 / nb * invR);
    } else {
      acc += a0 * a0 + a1 * a1 + b0 * b0 + b1 * b1;
      d = make_float4(-2.f * a0 * invR, -2.f * a1 * invR, -2.f * b0 * invR, -2.f * b1 * invR);
    }
    if (dmu) reinterpret_cast<float4*>(dmu)[q] = d;
  }
  if ((R & 1) && blockIdx.x == 0 && threadIdx.x == 0)
    acc += loss_row(mu + (R - 1) * 2, y + (R - 1) * 2, dmu ? dmu + (R - 1) * 2 : nullptr, 2, kind, invR);
  loss_finish(acc, red, &last, loss, invR);
}
extern "C" int b200np_loss_fwd_bwd(const float* mu, const float* y, float* loss, float* dmu, long long R,
                                   int out, int L, int kind, void* stream) {
  if (!mu || !y || !loss || R <= 0) return B200NP_E_BADARG;
  if (kind == 0 && (out != 2 || L < 2)) return B200NP_E_BADARG;
  if (kind == 1 && (out != 4 || L != 4)) return B200NP_E_BADARG;
  if (kind == 2 && (out != 2 || L < 2)) return B200NP_E_BADARG;
  if (kind == 3 && (out != 2 || L < 1 || dmu)) return B200NP_E_BADARG;
  if (kind < 0 || kind > 3) return B200NP_E_BADARG;
  if (R > 16384) {
    long long blocks = ceil_div(R, 256 * 4);
    if (blocks > kLossBlocks) blocks = kLossBlocks;
    if ((kind == 0 || kind == 2) && L == 2 && aligned16(mu) && aligned16(y) && (!dmu || aligned16(dmu)))
      loss_multi_vec_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(mu, y, loss, dmu, R, kind);
    else
      loss_multi_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(mu, y, loss, dmu, R, out, L, kind);
    return launch_status();
  }
  loss_kernel<<<1, 1024, 0, as_stream(stream)>>>(mu, y, loss, dmu, R, out, L, kind);
  return launch_status();
}

// ------------------------------------------------------------------------------------------------
// Total gradient norm over a flat segment: out = scale * ||g||_2.  A grid that depends on n only, per-thread fp64 sums in
// a fixed order, fixed-shape block trees, and a one-block second stage over the partials in the caller's workspace: the
// result is bitwise repeatable, and two calls with different workspaces may run concurrently.  fp64 sums of squares of
// finite fp32 values cannot overflow, so the result is finite exactly when every element is.
// ------------------------------------------------------------------------------------------------
constexpr int kNormThreads = 256;
constexpr long long kNormBlocks = 4 * kNumSMs;
static long long norm_blocks(long long n) {
  long long b = ceil_div(ceil_div(n, 4), kNormThreads);
  return b < kNormBlocks ? b : kNormBlocks;
}
__device__ __forceinline__ double block_sum_f64(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) red[w] = v;
  __syncthreads();
  double t = lane < nw ? red[lane] : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  return t;
}
__global__ void __launch_bounds__(kNormThreads) grad_norm_partial_kernel(const float* __restrict__ g, long long n, int vec,
                                                                         double* __restrict__ part) {
  __shared__ double red[32];
  const long long st = (long long)gridDim.x * blockDim.x;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double acc = 0.0;
  long long tail = i;
  if (vec) {
    const long long n4 = n >> 2;
    for (long long k = i; k < n4; k += st) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(g) + k);
      acc = fma((double)x.x, (double)x.x, acc);
      acc = fma((double)x.y, (double)x.y, acc);
      acc = fma((double)x.z, (double)x.z, acc);
      acc = fma((double)x.w, (double)x.w, acc);
    }
    tail = (n4 << 2) + i;
  }
  for (long long k = tail; k < n; k += st) {
    const double x = __ldg(g + k);
    acc = fma(x, x, acc);
  }
  acc = block_sum_f64(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(kNormThreads) grad_norm_finish_kernel(const double* __restrict__ part, int nparts,
                                                                        float scale, float* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int b = threadIdx.x; b < nparts; b += blockDim.x) s += part[b];
  s = block_sum_f64(s, red);
  if (threadIdx.x == 0) {
    const double r = sqrt(s) * (double)scale;
    // a finite norm beyond the fp32 range saturates, so that out[0] is finite exactly when every element is
    out[0] = isfinite(r) ? (float)fmin(r, (double)FLT_MAX) : (float)r;
  }
}
extern "C" size_t b200np_grad_norm_workspace(long long n) {
  return n > 0 ? (size_t)norm_blocks(n) * sizeof(double) : 0;
}
extern "C" int b200np_grad_norm(const float* g, long long n, float scale, float* out, void* ws, size_t ws_bytes,
                                void* stream) {
  if (!g || !out || n <= 0) return B200NP_E_BADARG;
  if (!ws || ws_bytes < b200np_grad_norm_workspace(n)) return B200NP_E_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) & 7u) return B200NP_E_BADARG;
  const long long blocks = norm_blocks(n);
  double* part = static_cast<double*>(ws);
  grad_norm_partial_kernel<<<(unsigned)blocks, kNormThreads, 0, as_stream(stream)>>>(g, n, aligned16(g), part);
  grad_norm_finish_kernel<<<1, kNormThreads, 0, as_stream(stream)>>>(part, (int)blocks, scale, out);
  return launch_status(2);
}

// ------------------------------------------------------------------------------------------------
// Fused Adam on a flat segment: 16 B read + 12 B written per parameter, float4 vectorised.
// One kernel serves every entry point.  Its hyperparameters come from a group table (b200np_adam_step_groups) or from
// one group passed by value (the single-group entry points); each block derives the per-group bias corrections once
// into shared memory.  A block updates one contiguous range of the segment, so the run table (which run of the
// segment belongs to which group) is searched once per thread and then walked forward.
// ------------------------------------------------------------------------------------------------
struct AdamHyper {
  float step_size, inv_bc2_sqrt, b1, b2, eps;
  float wd;     // coupled (L2) decay, folded into the gradient; 0 with decoupled decay
  float decay;  // decoupled (AdamW) decay: p *= decay before the update; 1 otherwise
};
__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamHyper& h, float gs) {
  g *= gs;
  if (h.decay != 1.f) p *= h.decay;
  if (h.wd != 0.f) g = fmaf(h.wd, p, g);
  m = m + (g - m) * (1.f - h.b1);
  v = v * h.b2 + (1.f - h.b2) * g * g;
  float denom = sqrtf(v) * h.inv_bc2_sqrt + h.eps;
  p = p - h.step_size * (m / denom);
}
__device__ __forceinline__ AdamHyper adam_hyper(const b200np_adam_group& G, const int* step_dev, float step_size,
                                                float inv_bc2_sqrt) {
  AdamHyper h{step_size, inv_bc2_sqrt, G.beta1, G.beta2, G.eps, G.decoupled ? 0.f : G.weight_decay, 1.f};
  if (step_dev) {  // CUDA-graph friendly: the step count lives on the device, bias corrections are derived here
    const double t = (double)__ldg(step_dev);
    h.step_size = (float)((double)G.lr / (1.0 - pow((double)G.beta1, t)));
    h.inv_bc2_sqrt = (float)(1.0 / sqrt(1.0 - pow((double)G.beta2, t)));
  }
  if (G.decoupled) h.decay = (float)(1.0 - (double)G.lr * (double)G.weight_decay);
  return h;
}
__device__ __forceinline__ bool adam_skips(const float* norm, bool skip) { return skip && !isfinite(__ldg(norm)); }
// the step counter ticks unless the step is skipped; a skipped step ticks `skipped` instead
__global__ void adam_tick_kernel(int* step, const float* norm, int* skipped) {
  if (adam_skips(norm, skipped != nullptr))
    *skipped += 1;
  else
    *step += 1;
}

constexpr int kAdamThreads = 256;
constexpr int kAdamMaxGroups = 1024;  // shared memory per block: kAdamMaxGroups * sizeof(AdamHyper)
struct AdamArgs {
  float* p;
  const float* g;
  float* m;
  float* v;
  long long n;
  int vec;                          // every pointer 16-B aligned: float4 units, else single floats
  float gs;                         // gradient scale (1/world)
  const int* step_dev;              // nullable: the host bias corrections below are used
  float step_size, inv_bc2_sqrt;
  const b200np_adam_group* groups;  // nullable: one group, `one`, over [0, n)
  int n_groups, n_runs;
  const long long* run_begin;       // n_runs + 1 float offsets, multiples of 4, from 0 to n
  const int* run_group;             // group of each run, -1: frozen
  b200np_adam_group one;
  const float* lr_dev;              // one group: nullable, replaces one.lr
  const float* max_norm;            // nullable: no clipping
  const float* norm;                // b200np_grad_norm of the same (grad_scale-scaled) gradient
  int skip;                         // leave everything unchanged when *norm is not finite
};

// the group of run r; a group index outside the table counts as frozen, so a bad table never reads past `hyp`
__device__ __forceinline__ int adam_run_group(const AdamArgs& a, int r, int ng) {
  const int grp = __ldg(a.run_group + r);
  return grp < ng ? grp : -1;
}

__global__ void __launch_bounds__(kAdamThreads) adam_kernel(const AdamArgs a) {
  extern __shared__ AdamHyper hyp[];
  if (adam_skips(a.norm, a.skip)) return;
  float gs = a.gs;
  if (a.max_norm) {
    // torch.nn.utils.clip_grad_norm_'s coefficient, NaN included; folded into the scale, which it leaves unchanged
    // when it is 1
    const float c = __ldg(a.max_norm) / (__ldg(a.norm) + 1e-6f);
    gs *= c >= 1.f ? 1.f : c;
  }
  const int ng = a.groups ? a.n_groups : 1;
  for (int i = threadIdx.x; i < ng; i += blockDim.x) {
    b200np_adam_group G = a.groups ? a.groups[i] : a.one;
    if (!a.groups && a.lr_dev) G.lr = __ldg(a.lr_dev);
    hyp[i] = adam_hyper(G, a.step_dev, a.step_size, a.inv_bc2_sqrt);
  }
  __syncthreads();

  const long long nu = a.vec ? a.n >> 2 : a.n;
  const long long bx = blockDim.x, per = ((nu + gridDim.x - 1) / gridDim.x + bx - 1) / bx * bx;
  const long long lo = (long long)blockIdx.x * per, hi = lo + per < nu ? lo + per : nu;
  long long k = lo + threadIdx.x;
  // the run holding unit k: [run_begin[r], run_begin[r + 1]) in floats, `end` in units
  int r = 0, grp = 0;
  long long end = nu;
  if (a.run_begin && k < hi) {
    int l = 0, u = a.n_runs - 1;
    while (l < u) {
      const int mid = (l + u + 1) >> 1;
      if (__ldg(a.run_begin + mid) <= 4 * k) l = mid; else u = mid - 1;
    }
    r = l;
    end = __ldg(a.run_begin + r + 1) >> 2;
    grp = adam_run_group(a, r, ng);
  }
  AdamHyper h = hyp[grp < 0 ? 0 : grp];
  for (; k < hi; k += blockDim.x) {
    if (k >= end) {
      do end = __ldg(a.run_begin + (++r) + 1) >> 2; while (k >= end);
      grp = adam_run_group(a, r, ng);
      if (grp >= 0) h = hyp[grp];
    }
    if (grp < 0) continue;  // frozen: neither read nor written
    if (a.vec) {
      float4 P = reinterpret_cast<float4*>(a.p)[k], G = reinterpret_cast<const float4*>(a.g)[k];
      float4 M = reinterpret_cast<float4*>(a.m)[k], V = reinterpret_cast<float4*>(a.v)[k];
      adam_one(P.x, G.x, M.x, V.x, h, gs);
      adam_one(P.y, G.y, M.y, V.y, h, gs);
      adam_one(P.z, G.z, M.z, V.z, h, gs);
      adam_one(P.w, G.w, M.w, V.w, h, gs);
      reinterpret_cast<float4*>(a.p)[k] = P;
      reinterpret_cast<float4*>(a.m)[k] = M;
      reinterpret_cast<float4*>(a.v)[k] = V;
    } else {
      adam_one(a.p[k], a.g[k], a.m[k], a.v[k], h, gs);
    }
  }
  // the scalar tail of a float4 segment (one group only: a run table needs n % 4 == 0)
  if (a.vec && blockIdx.x == gridDim.x - 1)
    for (long long t = (nu << 2) + threadIdx.x; t < a.n; t += blockDim.x)
      adam_one(a.p[t], a.g[t], a.m[t], a.v[t], hyp[0], gs);
}

// tick (when `step_dev`) + update; `a` carries everything but the launch shape
static int adam_launch(AdamArgs a, int* step_dev, int* skipped, void* stream) {
  a.vec = aligned16(a.p) && aligned16(a.g) && aligned16(a.m) && aligned16(a.v);
  a.step_dev = step_dev;
  a.skip = skipped != nullptr;
  const size_t smem = (size_t)(a.groups ? a.n_groups : 1) * sizeof(AdamHyper);
  if (step_dev) adam_tick_kernel<<<1, 1, 0, as_stream(stream)>>>(step_dev, a.norm, skipped);
  adam_kernel<<<ew_grid((a.n + 3) / 4, kAdamThreads), kAdamThreads, smem, as_stream(stream)>>>(a);
  return launch_status(step_dev ? 2 : 1);
}

extern "C" int b200np_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr,
                                float beta1, float beta2, float eps, float weight_decay, int step,
                                float grad_scale, void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!p || !g || !m || !v || step < 1) return B200NP_E_BADARG;
  double bc1 = 1.0 - pow((double)beta1, (double)step);
  double bc2 = 1.0 - pow((double)beta2, (double)step);
  AdamArgs a{};
  a.p = p, a.g = g, a.m = m, a.v = v, a.n = n, a.gs = grad_scale;
  a.step_size = (float)((double)lr / bc1);
  a.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
  a.one = b200np_adam_group{lr, weight_decay, beta1, beta2, eps, 0};
  return adam_launch(a, nullptr, nullptr, stream);
}

extern "C" int b200np_adam_step_dev(float* p, const float* g, float* m, float* v, long long n, float lr,
                                    float beta1, float beta2, float eps, float weight_decay, int* step_dev,
                                    float grad_scale, void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!p || !g || !m || !v || !step_dev) return B200NP_E_BADARG;
  AdamArgs a{};
  a.p = p, a.g = g, a.m = m, a.v = v, a.n = n, a.gs = grad_scale;
  a.one = b200np_adam_group{lr, weight_decay, beta1, beta2, eps, 0};
  return adam_launch(a, step_dev, nullptr, stream);
}

extern "C" int b200np_adam_step_ctrl(float* p, const float* g, float* m, float* v, long long n, const float* lr,
                                     float beta1, float beta2, float eps, float weight_decay, int* step_dev,
                                     float grad_scale, const float* max_norm, const float* norm, int* skipped,
                                     void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!p || !g || !m || !v || !lr || !step_dev || ((max_norm || skipped) && !norm)) return B200NP_E_BADARG;
  AdamArgs a{};
  a.p = p, a.g = g, a.m = m, a.v = v, a.n = n, a.gs = grad_scale;
  a.one = b200np_adam_group{0.f, weight_decay, beta1, beta2, eps, 0};
  a.lr_dev = lr, a.max_norm = max_norm, a.norm = norm;
  return adam_launch(a, step_dev, skipped, stream);
}

extern "C" int b200np_adam_step_groups(float* p, const float* g, float* m, float* v, long long n,
                                       const b200np_adam_group* groups, int n_groups, const long long* run_begin,
                                       const int* run_group, int n_runs, int* step_dev, float grad_scale,
                                       const float* max_norm, const float* norm, int* skipped, void* stream) {
  if (n <= 0) return B200NP_OK;
  if (!p || !g || !m || !v || !groups || !run_begin || !run_group || !step_dev || ((max_norm || skipped) && !norm))
    return B200NP_E_BADARG;
  if (n_groups < 1 || n_groups > kAdamMaxGroups || n_runs < 1 || n % 4) return B200NP_E_BADARG;
  if (!aligned16(p) || !aligned16(g) || !aligned16(m) || !aligned16(v)) return B200NP_E_BADARG;
  AdamArgs a{};
  a.p = p, a.g = g, a.m = m, a.v = v, a.n = n, a.gs = grad_scale;
  a.groups = groups, a.n_groups = n_groups, a.run_begin = run_begin, a.run_group = run_group, a.n_runs = n_runs;
  a.max_norm = max_norm, a.norm = norm;
  return adam_launch(a, step_dev, skipped, stream);
}
