// Condition adapters of UNetSD_VideoLCM / UNetSD_TFT2V (unet_videolcm.py:294-372, forward :598-703).
//
// Every adapter starts with Conv2d(cin -> Cout, 3x3, pad 1) -> SiLU -> AdaptiveAvgPool2d(resolution / 2) on the condition
// at full pixel resolution, once per frame.  vgen_cond_stem does the three in one pass: a CTA stages a halo tile of the
// condition (read in the reference layout [b, cin, f, H, W], fp32 or fp16) in shared memory, builds the im2col
// fragments of a 16 x 32 pre-pool region from it, runs the MACs on the tensor cores (mma.sync m16n8k16, K = 9*cin
// padded to 16 / 32 / 48), keeps the SiLU'd conv tile in shared memory and writes only the pooled result.  The output
// tiles are chosen on the host so that every pooling window of a CTA lies inside its region: neither the Cout-channel
// full-resolution tensor nor any im2col column reaches HBM.
//
// Rounding follows the reference under fp16 autocast: the condition is rounded to fp16 (autocast's input cast), the
// conv result (fp32 accumulation + fp32 bias) is rounded to fp16, SiLU runs in fp32 on that value and is rounded to
// fp16, the pool sums in fp32 and rounds the mean to fp16.
//
// vgen_cond_sum adds the adapter outputs in fp32 in the caller's order and rounds once (the reference accumulates into
// the fp32 `concat = x.new_zeros(...)`, :598-699).
#include <algorithm>

#include "common.h"

namespace vg {
namespace {

constexpr int kRH = 16;                  // pre-pool rows per CTA
constexpr int kRW = 32;                  // pre-pool columns per CTA
constexpr int kHR = kRH + 2;             // halo tile rows
constexpr int kHC = kRW + 2;             // halo tile columns
constexpr int kMaxCin = 4;
constexpr int kZeroBase = kMaxCin * kHR * kHC;                       // padded im2col columns read a zero band here
constexpr int kHaloElems = kZeroBase + kHR * kHC;                      // the band is longer than any pixel offset
constexpr int kStemThreads = 256;

__device__ __forceinline__ float silu_f(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

__device__ __forceinline__ void mma_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t pack_h2(__half lo, __half hi) {
  return (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
}

// KS k-steps of 16 (K = 9*cin padded), NT n-tiles of 8 output channels.
template <typename T, int KS, int NT>
__global__ void __launch_bounds__(kStemThreads) cond_stem_kernel(const T* __restrict__ x, const __half* __restrict__ wt,
                                                                 const float* __restrict__ bias, __half* __restrict__ out,
                                                                 int cin, int f, int H, int W, int oh, int ow, int toh,
                                                                 int tow, int tiles_w) {
  constexpr int COUT = NT * 8;
  constexpr int KP = KS * 16;
  constexpr int CST = COUT + 8;          // conv-tile row stride in halves (+8: conflict-free half2 stores)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* halo = reinterpret_cast<__half*>(smem_raw);           // [cin][kHR][kHC] ... zero band at kZeroBase
  __half* conv = halo + kHaloElems;                             // [kRH * kRW][CST]

  const int img = blockIdx.y;
  const int ti = blockIdx.x / tiles_w, tj = blockIdx.x % tiles_w;
  const int i0 = ti * toh, j0 = tj * tow;
  const int i1 = min(i0 + toh, oh), j1 = min(j0 + tow, ow);
  // pre-pool region of this tile: the union of its adaptive pooling windows (torch: [floor(i*in/out), ceil((i+1)*in/out)))
  const int r0 = (int)(((long)i0 * H) / oh), r1 = (int)(((long)i1 * H + oh - 1) / oh);
  const int c0 = (int)(((long)j0 * W) / ow);

  // ---- halo tile of the condition (fp16, zero outside the image = the conv's padding)
  const int b = img / f, fi = img % f;
  const long plane = (long)H * W;
  const T* xb = x + ((long)b * cin * f + fi) * plane;
  const int nh = cin * kHR * kHC;
  for (int e = threadIdx.x; e < nh; e += kStemThreads) {
    const int ci = e / (kHR * kHC), rem = e - ci * (kHR * kHC);
    const int gr = r0 - 1 + rem / kHC, gc = c0 - 1 + rem % kHC;
    float v = 0.f;
    if (gr >= 0 && gr < H && gc >= 0 && gc < W) v = (float)xb[(long)ci * f * plane + (long)gr * W + gc];
    halo[e] = __float2half_rn(v);
  }
  for (int e = threadIdx.x; e < kHR * kHC; e += kStemThreads) halo[kZeroBase + e] = __float2half_rn(0.f);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tig = lane & 3;

  // this thread's im2col column offsets into the halo: k = tap*cin + ci, tap = ky*3 + kx; padded k -> the zero band
  int koff[KS][4];
#pragma unroll
  for (int s = 0; s < KS; ++s)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int k = s * 16 + (q >> 1) * 8 + tig * 2 + (q & 1);
      const int tap = k / cin, ci = k - tap * cin;
      koff[s][q] = k < 9 * cin ? ci * (kHR * kHC) + (tap / 3) * kHC + (tap % 3) : kZeroBase;
    }
  // B fragments (weights, K-major [COUT][KP]) and bias stay in registers for the whole CTA
  uint32_t bf[KS][NT][2];
  float bs[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const __half* wr = wt + (long)(nt * 8 + g) * KP + tig * 2;
#pragma unroll
    for (int s = 0; s < KS; ++s) {
      bf[s][nt][0] = *reinterpret_cast<const uint32_t*>(wr + s * 16);
      bf[s][nt][1] = *reinterpret_cast<const uint32_t*>(wr + s * 16 + 8);
    }
    bs[nt][0] = bias[nt * 8 + tig * 2];
    bs[nt][1] = bias[nt * 8 + tig * 2 + 1];
  }
  __syncthreads();

  // ---- conv + bias + SiLU on the region: m-tiles of 16 pixels (half a region row), 4 per warp
  const int rows = r1 - r0;
  for (int mt = warp; mt < (kRH * kRW) / 16; mt += kStemThreads / 32) {
    const int pr = (mt * 16) / kRW;
    if (pr >= rows) break;                                   // warp-uniform
    const int pc = (mt * 16) % kRW + g;                      // rows g and g + 8 of the m-tile
    const int base0 = pr * kHC + pc, base1 = base0 + 8;
    uint32_t a[KS][4];
#pragma unroll
    for (int s = 0; s < KS; ++s) {
      __half v0[4], v1[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        v0[q] = halo[base0 + koff[s][q]];
        v1[q] = halo[base1 + koff[s][q]];
      }
      a[s][0] = pack_h2(v0[0], v0[1]);   // row g,     k = tig*2 + {0,1}
      a[s][1] = pack_h2(v1[0], v1[1]);   // row g + 8
      a[s][2] = pack_h2(v0[2], v0[3]);   // row g,     k = 8 + tig*2 + {0,1}
      a[s][3] = pack_h2(v1[2], v1[3]);   // row g + 8
    }
    float acc[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
      for (int s = 0; s < KS; ++s) mma_16816(acc[nt], a[s], bf[s][nt][0], bf[s][nt][1]);
    }
    __half* c0p = conv + (pr * kRW + pc) * CST + tig * 2;
    __half* c1p = c0p + 8 * CST;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float h = __half2float(__float2half_rn(acc[nt][q] + bs[nt][q & 1]));   // conv output, fp16
        v[q] = silu_f(h);
      }
      *reinterpret_cast<__half2*>(c0p + nt * 8) = __floats2half2_rn(v[0], v[1]);
      *reinterpret_cast<__half2*>(c1p + nt * 8) = __floats2half2_rn(v[2], v[3]);
    }
  }
  __syncthreads();

  // ---- adaptive average pool of the tile: fp32 sums (row-major over the window), mean rounded to fp16
  const int tw = j1 - j0;
  const int n_out = (i1 - i0) * tw * (COUT / 2);
  for (int e = threadIdx.x; e < n_out; e += kStemThreads) {
    const int cp = e % (COUT / 2), q = e / (COUT / 2);
    const int oi = i0 + q / tw, oj = j0 + q % tw;
    const int ys = (int)(((long)oi * H) / oh), ye = (int)(((long)(oi + 1) * H + oh - 1) / oh);
    const int xs = (int)(((long)oj * W) / ow), xe = (int)(((long)(oj + 1) * W + ow - 1) / ow);
    float sx = 0.f, sy = 0.f;
    for (int rr = ys; rr < ye; ++rr)
      for (int cc = xs; cc < xe; ++cc) {
        const float2 v = __half22float2(*reinterpret_cast<const __half2*>(conv + ((rr - r0) * kRW + (cc - c0)) * CST + cp * 2));
        sx += v.x;
        sy += v.y;
      }
    const float cnt = (float)((ye - ys) * (xe - xs));
    *reinterpret_cast<__half2*>(out + (((long)img * oh + oi) * ow + oj) * COUT + cp * 2) = __floats2half2_rn(sx / cnt, sy / cnt);
  }
}

// Largest output tile along one axis whose pooling windows all fit a region of `rmax` input positions.
int pick_tile(long in, long out, int rmax) {
  for (long t = std::min<long>(out, rmax); t >= 1; --t) {
    bool ok = true;
    for (long i0 = 0; i0 < out && ok; i0 += t) {
      const long i1 = std::min(i0 + t, out);
      ok = ((i1 * in + out - 1) / out) - (i0 * in) / out <= rmax;
    }
    if (ok) return (int)t;
  }
  return 0;
}

template <typename T, int KS, int NT>
int launch_stem(const void* x, const void* wt, const float* bias, void* out, long nimg, int cin, int f, int H, int W, int oh,
                int ow, int toh, int tow, cudaStream_t stream) {
  constexpr int CST = NT * 8 + 8;
  const size_t smem = (size_t)(kHaloElems + kRH * kRW * CST) * sizeof(__half);
  if (smem > 48 * 1024) {
    static PerDeviceOnce once;
    if (once.need()) {
      VG_CUDA(cudaFuncSetAttribute(cond_stem_kernel<T, KS, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      once.mark();
    }
  }
  const int tiles_w = (ow + tow - 1) / tow;
  const int tiles = ((oh + toh - 1) / toh) * tiles_w;
  launch_kernel(cond_stem_kernel<T, KS, NT>, dim3((unsigned)tiles, (unsigned)nimg), dim3(kStemThreads), smem, stream,
                reinterpret_cast<const T*>(x), reinterpret_cast<const __half*>(wt), bias, reinterpret_cast<__half*>(out),
                cin, f, H, W, oh, ow, toh, tow, tiles_w);
  VG_LAUNCH_CHECK("cond_stem_kernel");
  return 0;
}

template <typename T, int KS>
int dispatch_nt(int nt, const void* x, const void* wt, const float* bias, void* out, long nimg, int cin, int f, int H, int W,
                int oh, int ow, int toh, int tow, cudaStream_t s) {
  switch (nt) {
#define VG_STEM_NT(N) \
  case N: return launch_stem<T, KS, N>(x, wt, bias, out, nimg, cin, f, H, W, oh, ow, toh, tow, s);
    VG_STEM_NT(1) VG_STEM_NT(2) VG_STEM_NT(3) VG_STEM_NT(4) VG_STEM_NT(5) VG_STEM_NT(6) VG_STEM_NT(7) VG_STEM_NT(8)
#undef VG_STEM_NT
  }
  return fail("vgen_cond_stem: cout must be 8..64 in steps of 8");
}

template <typename T>
int dispatch_ks(int ks, int nt, const void* x, const void* wt, const float* bias, void* out, long nimg, int cin, int f, int H,
                int W, int oh, int ow, int toh, int tow, cudaStream_t s) {
  switch (ks) {
    case 1: return dispatch_nt<T, 1>(nt, x, wt, bias, out, nimg, cin, f, H, W, oh, ow, toh, tow, s);
    case 2: return dispatch_nt<T, 2>(nt, x, wt, bias, out, nimg, cin, f, H, W, oh, ow, toh, tow, s);
    case 3: return dispatch_nt<T, 3>(nt, x, wt, bias, out, nimg, cin, f, H, W, oh, ow, toh, tow, s);
  }
  return fail("vgen_cond_stem: cin must be 1..4");
}

constexpr int kMaxSum = 8;
struct SumSrcs {
  const __half* p[kMaxSum];
};

__global__ void cond_sum_kernel(SumSrcs src, int nsrc, long rows, int cols, long ld_src, __half* __restrict__ out, long ld_out) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  const long r = idx / cols;
  const int c = (int)(idx - r * cols);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxSum; ++i)
    if (i < nsrc) s += __half2float(src.p[i][r * ld_src + c]);
  out[r * ld_out + c] = __float2half_rn(s);
}

}  // namespace
}  // namespace vg

using namespace vg;

extern "C" {

int vgen_cond_stem(const void* x, int x_is_f32, int64_t b, int64_t cin, int64_t f, int64_t h, int64_t w, const void* wt,
                   const float* bias, int64_t cout, int64_t oh, int64_t ow, void* out, void* stream) {
  VG_REQUIRE(x && wt && bias && out, "vgen_cond_stem: null pointer");
  VG_REQUIRE(b > 0 && f > 0 && h > 0 && w > 0 && oh > 0 && ow > 0, "vgen_cond_stem: bad shape");
  VG_REQUIRE(cin >= 1 && cin <= kMaxCin, "vgen_cond_stem: cin must be 1..4");
  VG_REQUIRE(cout >= 8 && cout <= 64 && cout % 8 == 0, "vgen_cond_stem: cout must be 8..64 in steps of 8");
  VG_REQUIRE(b * f <= 65535, "vgen_cond_stem: b*f must be <= 65535");
  VG_REQUIRE(h * w < (1ll << 31) && oh * ow < (1ll << 31), "vgen_cond_stem: image too large");
  const int toh = pick_tile(h, oh, kRH), tow = pick_tile(w, ow, kRW);
  VG_REQUIRE(toh > 0 && tow > 0, "vgen_cond_stem: a pooling window spans more than 16 rows or 32 columns");
  const int ks = (int)((9 * cin + 15) / 16);
  const cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (x_is_f32)
    return dispatch_ks<float>(ks, (int)(cout / 8), x, wt, bias, out, b * f, (int)cin, (int)f, (int)h, (int)w, (int)oh, (int)ow,
                              toh, tow, s);
  return dispatch_ks<__half>(ks, (int)(cout / 8), x, wt, bias, out, b * f, (int)cin, (int)f, (int)h, (int)w, (int)oh, (int)ow,
                             toh, tow, s);
}

int vgen_cond_sum(const void* const* srcs, int nsrc, int64_t rows, int64_t cols, int64_t ld_src, void* out, int64_t ld_out,
                  void* stream) {
  VG_REQUIRE(srcs && out && nsrc >= 1 && nsrc <= kMaxSum, "vgen_cond_sum: 1..8 sources");
  VG_REQUIRE(rows >= 0 && cols > 0 && ld_src >= cols && ld_out >= cols, "vgen_cond_sum: bad shape");
  SumSrcs p = {};
  for (int i = 0; i < nsrc; ++i) {
    VG_REQUIRE(srcs[i], "vgen_cond_sum: null source");
    p.p[i] = reinterpret_cast<const __half*>(srcs[i]);
  }
  const long total = rows * cols;
  if (total == 0) return 0;
  launch_kernel(cond_sum_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p,
                nsrc, (long)rows, (int)cols, (long)ld_src, reinterpret_cast<__half*>(out), (long)ld_out);
  VG_LAUNCH_CHECK("cond_sum_kernel");
  return 0;
}

}  // extern "C"
