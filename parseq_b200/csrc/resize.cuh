// Batched ragged bicubic resize of RGB uint8 crops to the engine's uint8 HWC input [N, img_h, img_w, 3]: the
// reference's `img.rotate(rotation, expand=True)` + `T.Resize(img_size, BICUBIC)` on PIL images
// (strhub/data/module.py:69-82), bit-exact with PIL's resampler (libImaging/Resample.c):
//   - coefficients per output index in double precision with precompute_coeffs' expression order (bicubic, a = -0.5),
//     built from __dadd_rn / __dmul_rn / __ddiv_rn so that nothing is contracted into an FMA, truncating conversions
//     where C casts, then quantised to int32 with 22 fraction bits (round half away from zero);
//   - integer sums seeded with 2^21, clipped to uint8 after each pass;
//   - horizontal pass first, except for crops more than 100 times taller than wide that shrink vertically, which
//     Image.resize resizes height first; an axis whose size does not change is copied, not resampled.
// Rotation by 0 / 90 / 180 / 270 degrees (counter-clockwise, expand=True: an exact transpose) is folded into the
// source indexing of the first pass.
//
// One CTA per task = (crop, band of output rows, tile of output columns), planned on the host so that the task's
// shared memory fits.  Horizontal-first: the first pass writes the window of source rows the band's vertical taps
// touch, resampled to the tile's columns, into shared memory as uint8; the second pass resamples it vertically into
// the band.  Vertical-first: the first pass writes the band's rows at the full source width, the second resamples
// them horizontally into the tile.
#pragma once
#include "ptx.cuh"

namespace pq {

constexpr int RZ_PRECISION_BITS = 22;
constexpr int RZ_THREADS = 256;

struct RzCrop {
  long long offset;   // byte offset of pixel (0, 0) in the packed buffer
  int h, w, stride;   // source size (before rotation) and row stride in bytes
  int hr, wr;         // size after rotation
  int vfirst;         // 1: vertical pass first
};

struct RzTask {
  int crop;
  int y0, ny;         // output rows of the band
  int x0, nx;         // output columns of the tile
  int r0, nr;         // window rows held in shared memory: source rows (horizontal first) / output rows (vertical first)
};

// filter geometry of one axis: in_size -> out_size (precompute_coeffs)
struct RzAxis {
  double scale, support, ss;
  int ksize;
};

__host__ __device__ inline int rz_ksize(int in_size, int out_size) {
  const double scale = static_cast<double>(in_size) / out_size;
  const double fs = scale < 1.0 ? 1.0 : scale;
  return static_cast<int>(ceil(2.0 * fs)) * 2 + 1;
}

__device__ __forceinline__ RzAxis rz_axis(int in_size, int out_size) {
  RzAxis a;
  a.scale = __ddiv_rn(static_cast<double>(in_size), static_cast<double>(out_size));
  const double fs = a.scale < 1.0 ? 1.0 : a.scale;
  a.support = __dmul_rn(2.0, fs);
  a.ss = __ddiv_rn(1.0, fs);
  a.ksize = static_cast<int>(ceil(a.support)) * 2 + 1;
  return a;
}

// bicubic_filter, a = -0.5:  |x| < 1: ((a + 2) x - (a + 3)) x x + 1;  |x| < 2: (((x - 5) x + 8) x - 4) a
__device__ __forceinline__ double rz_bicubic(double x) {
  if (x < 0.0) x = -x;
  if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);
  if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
  return 0.0;
}

// Taps of output index xx: first source index -> *xmin, tap count -> *cnt, quantised weights -> k[0 .. cnt).
__device__ void rz_coeffs(const RzAxis& a, int in_size, int xx, int* xmin_out, int* cnt_out, int* k) {
  const double center = __dmul_rn(__dadd_rn(static_cast<double>(xx), 0.5), a.scale);
  int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, a.support), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, a.support), 0.5));
  if (xmax > in_size) xmax = in_size;
  xmax -= xmin;
  double ww = 0.0;
  for (int x = 0; x < xmax; ++x)
    ww = __dadd_rn(ww, rz_bicubic(__dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(x + xmin), center), 0.5), a.ss)));
  for (int x = 0; x < xmax; ++x) {
    double w = rz_bicubic(__dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(x + xmin), center), 0.5), a.ss));
    if (ww != 0.0) w = __ddiv_rn(w, ww);
    const double q = __dmul_rn(w, static_cast<double>(1 << RZ_PRECISION_BITS));
    k[x] = __double2int_rz(w < 0.0 ? __dadd_rn(-0.5, q) : __dadd_rn(0.5, q));
  }
  *xmin_out = xmin;
  *cnt_out = xmax;
}

__device__ __forceinline__ uint8_t rz_clip8(int acc) {
  const int v = acc >> RZ_PRECISION_BITS;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// Pixel (yr, xr) of the rotated crop (np.rot90 by rot / 90, as PIL's rotate(expand=True)).
__device__ __forceinline__ const uint8_t* rz_src(const uint8_t* base, const RzCrop& c, int rot, int yr, int xr) {
  int y = yr, x = xr;
  if (rot == 90) { y = xr; x = c.w - 1 - yr; }
  else if (rot == 180) { y = c.h - 1 - yr; x = c.w - 1 - xr; }
  else if (rot == 270) { y = c.h - 1 - xr; x = yr; }
  return base + static_cast<long long>(y) * c.stride + 3 * x;
}

__global__ void __launch_bounds__(RZ_THREADS) resize_bicubic_u8_kernel(const uint8_t* __restrict__ pixels,
                                                                       const RzCrop* __restrict__ crops,
                                                                       const RzTask* __restrict__ tasks, int crop_base,
                                                                       uint8_t* __restrict__ out, int H, int W, int rot) {
  grid_dep_launch();
  extern __shared__ __align__(16) unsigned char rz_smem[];
  const RzTask t = tasks[blockIdx.x];
  const RzCrop c = crops[t.crop];
  const uint8_t* base = pixels + c.offset;
  const bool need_h = c.wr != W, need_v = c.hr != H;
  const RzAxis ah = rz_axis(c.wr, W), av = rz_axis(c.hr, H);
  const int kh = need_h ? ah.ksize : 0, kv = need_v ? av.ksize : 0;
  // shared memory: [ny + nx] bounds pairs, [ny][kv] + [nx][kh] weights, then the uint8 window
  int* vb = reinterpret_cast<int*>(rz_smem);          // [ny][2] vertical (xmin, cnt) of the band's rows
  int* hb = vb + 2 * t.ny;                             // [nx][2] horizontal of the tile's columns
  int* vk = hb + 2 * t.nx;                             // [ny][kv]
  int* hk = vk + t.ny * kv;                            // [nx][kh]
  uint8_t* win = reinterpret_cast<uint8_t*>(hk + t.nx * kh);
  const int wcols = c.vfirst ? c.wr : t.nx;            // window row width in pixels
  for (int i = threadIdx.x; i < t.ny; i += blockDim.x) {
    if (need_v) rz_coeffs(av, c.hr, t.y0 + i, &vb[2 * i], &vb[2 * i + 1], vk + i * kv);
    else { vb[2 * i] = t.y0 + i; vb[2 * i + 1] = 1; }
  }
  for (int j = threadIdx.x; j < t.nx; j += blockDim.x) {
    if (need_h) rz_coeffs(ah, c.wr, t.x0 + j, &hb[2 * j], &hb[2 * j + 1], hk + j * kh);
    else { hb[2 * j] = t.x0 + j; hb[2 * j + 1] = 1; }
  }
  __syncthreads();
  grid_dep_wait();                                     // the crops may be written by the previous kernel

  constexpr int HALF = 1 << (RZ_PRECISION_BITS - 1);
  // ---- first pass: source -> window
  const int n1 = t.nr * wcols;
  for (int e = threadIdx.x; e < n1; e += blockDim.x) {
    const int r = e / wcols, j = e - r * wcols;
    int s0 = HALF, s1 = HALF, s2 = HALF;
    if (!c.vfirst) {                                   // horizontal: window row = source row r0 + r, column = tile column j
      const int yr = t.r0 + r;
      if (!need_h) {
        const uint8_t* p = rz_src(base, c, rot, yr, t.x0 + j);
        win[e * 3 + 0] = p[0]; win[e * 3 + 1] = p[1]; win[e * 3 + 2] = p[2];
        continue;
      }
      const int x0 = hb[2 * j], n = hb[2 * j + 1];
      const int* k = hk + j * kh;
      for (int x = 0; x < n; ++x) {
        const uint8_t* p = rz_src(base, c, rot, yr, x0 + x);
        s0 += p[0] * k[x]; s1 += p[1] * k[x]; s2 += p[2] * k[x];
      }
    } else {                                           // vertical: window row = band row r, column = source column j
      const int y0 = vb[2 * r], n = vb[2 * r + 1];
      const int* k = vk + r * kv;
      for (int y = 0; y < n; ++y) {
        const uint8_t* p = rz_src(base, c, rot, y0 + y, j);
        s0 += p[0] * k[y]; s1 += p[1] * k[y]; s2 += p[2] * k[y];
      }
    }
    win[e * 3 + 0] = rz_clip8(s0); win[e * 3 + 1] = rz_clip8(s1); win[e * 3 + 2] = rz_clip8(s2);
  }
  __syncthreads();

  // ---- second pass: window -> band x tile of the output
  uint8_t* dst = out + static_cast<long long>(t.crop - crop_base) * H * W * 3;
  const int n2 = t.ny * t.nx;
  for (int e = threadIdx.x; e < n2; e += blockDim.x) {
    const int i = e / t.nx, j = e - i * t.nx;
    int s0 = HALF, s1 = HALF, s2 = HALF;
    uint8_t v0, v1, v2;
    if (!c.vfirst) {                                   // vertical over window rows (taps outside the window are skipped)
      const int y0 = vb[2 * i] - t.r0, n = vb[2 * i + 1];
      if (!need_v) {
        const uint8_t* p = win + (static_cast<long long>(y0) * wcols + j) * 3;
        v0 = p[0]; v1 = p[1]; v2 = p[2];
      } else {
        const int* k = vk + i * kv;
        for (int y = 0; y < n; ++y) {
          if (y0 + y < 0 || y0 + y >= t.nr) continue;
          const uint8_t* p = win + (static_cast<long long>(y0 + y) * wcols + j) * 3;
          s0 += p[0] * k[y]; s1 += p[1] * k[y]; s2 += p[2] * k[y];
        }
        v0 = rz_clip8(s0); v1 = rz_clip8(s1); v2 = rz_clip8(s2);
      }
    } else {                                           // horizontal over the band row's full source width
      const int x0 = hb[2 * j], n = hb[2 * j + 1];
      if (!need_h) {
        const uint8_t* p = win + (static_cast<long long>(i) * wcols + x0) * 3;
        v0 = p[0]; v1 = p[1]; v2 = p[2];
      } else {
        const int* k = hk + j * kh;
        const uint8_t* row = win + static_cast<long long>(i) * wcols * 3;
        for (int x = 0; x < n; ++x) {
          const uint8_t* p = row + (x0 + x) * 3;
          s0 += p[0] * k[x]; s1 += p[1] * k[x]; s2 += p[2] * k[x];
        }
        v0 = rz_clip8(s0); v1 = rz_clip8(s1); v2 = rz_clip8(s2);
      }
    }
    uint8_t* q = dst + (static_cast<long long>(t.y0 + i) * W + t.x0 + j) * 3;
    q[0] = v0; q[1] = v1; q[2] = v2;
  }
}

}  // namespace pq
