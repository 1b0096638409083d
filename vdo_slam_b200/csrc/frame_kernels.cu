// frame_kernels.cu -- image side of the per-frame path on sm_100a: depth pre-processing, ORB keypoints (pyramid, FAST score,
// per-cell FAST + NMS with threshold fallback, octree distribution, intensity-centroid angle), flow-guided static filter,
// semi-dense object sampling, back-projection and scene flow.
//
// Reference semantics (restated on the CPU in oracle/image_ops.py, with cv2 as the pin for the OpenCV-owned arithmetic):
//   depth pre-processing        src/Tracking.cc:180-204
//   ORBextractor                src/ORBextractor.cc:399-459, 754-842, 470-752, 66-93, 1035-1137
//   cv::resize (u8 INTER_LINEAR), cv::FAST (9/16, NMS), cv::fastAtan2: OpenCV (un-vendored); formulas verified bit-exact
//                               against cv2 4.13 in tests/test_image_oracle.py
//   Frame static filter         src/Frame.cc:100-129, 181-194
//   Frame object sampling       src/Frame.cc:200-228
//   sampled background keys     src/Frame.cc:672-740 (SampleKeyPoints, cv::RNG), 130-194 (Option II filter); restated in
//                               oracle/sampled_features.py
//   back-projection, scene flow src/Frame.cc:484-555, src/Tracking.cc:1278-1364
//
// A KITTI frame is 1242x375 (0.47 Mpx, ~9 MB of inputs): every kernel here is launch-/latency-bound, not HBM-bound; the
// point of the GPU path is to keep the frame resident next to the LM kernels, not bandwidth.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <list>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/vdo_b200.h"

namespace {

#define FRK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { std::fprintf(stderr, "[vdo_b200] CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return VDO_ERR_CUDA; } } while (0)

constexpr int EDGE_THRESHOLD = 19, PATCH_SIZE = 31, HALF_PATCH = 15, MAX_LEVELS = 12, CELL_CAP = 512;

// ------------------------------------------------------------------------------------------------ depth
__global__ void k_depth_prep(float* __restrict__ d, int n, float bf, float factor) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = d[i];
  d[i] = (v < 0.f) ? 0.f : (bf > 0.f ? __fdiv_rn(bf, __fdiv_rn(v, factor)) : v);   // mbf/(d/mDepthMapFactor), IEEE divisions (d == 0 -> +inf); bf <= 0: clamp only
}

// ------------------------------------------------------------------------------------------------ pyramid
// OpenCV u8 INTER_LINEAR: 11-bit fixed-point coefficients, horizontal pass in int, vertical pass with >>4, >>16, +2, >>2.
__device__ __forceinline__ void lin_coeff(int dpos, int sn, double scale, int& s0, int& s1, int& a0, int& a1) {
  float f = (float)((dpos + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (s < 0) { s = 0; f = 0.f; }
  if (s >= sn - 1) { s = sn - 1; f = 0.f; }
  s0 = s; s1 = min(s + 1, sn - 1);
  a0 = __float2int_rn((1.f - f) * 2048.f);
  a1 = __float2int_rn(f * 2048.f);
}
__global__ void k_resize_u8(const unsigned char* __restrict__ src, int sw, int sh, unsigned char* __restrict__ dst, int dw, int dh) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= dw || y >= dh) return;
  int x0, x1, ax0, ax1, y0, y1, ay0, ay1;
  lin_coeff(x, sw, (double)sw / dw, x0, x1, ax0, ax1);
  lin_coeff(y, sh, (double)sh / dh, y0, y1, ay0, ay1);
  const int h0 = src[(size_t)y0 * sw + x0] * ax0 + src[(size_t)y0 * sw + x1] * ax1;
  const int h1 = src[(size_t)y1 * sw + x0] * ax0 + src[(size_t)y1 * sw + x1] * ax1;
  int v = (((ay0 * (h0 >> 4)) >> 16) + ((ay1 * (h1 >> 4)) >> 16) + 2) >> 2;
  dst[(size_t)y * dw + x] = (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// ------------------------------------------------------------------------------------------------ FAST score
// score(p) = max over the 16 arcs of 9 contiguous circle pixels of min(|I_p - I_k| signed consistently) - 1
// (== cv::cornerScore<16>); a pixel is a FAST-9/16 corner at threshold t iff score >= t.
__global__ void k_fast_score(const unsigned char* __restrict__ img, int w, int h, unsigned char* __restrict__ score) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  int out = 0;
  if (x >= 3 && y >= 3 && x < w - 3 && y < h - 3) {
    const unsigned char* p = img + (size_t)y * w + x;
    const int v = p[0];
    // Bresenham circle of radius 3, clockwise from (0,+3); signed differences centre - neighbour
    int d[16];
    d[0] = v - p[3 * w];      d[1] = v - p[3 * w + 1];  d[2] = v - p[2 * w + 2];  d[3] = v - p[w + 3];
    d[4] = v - p[3];          d[5] = v - p[-w + 3];     d[6] = v - p[-2 * w + 2]; d[7] = v - p[-3 * w + 1];
    d[8] = v - p[-3 * w];     d[9] = v - p[-3 * w - 1]; d[10] = v - p[-2 * w - 2]; d[11] = v - p[-w - 3];
    d[12] = v - p[-3];        d[13] = v - p[w - 3];     d[14] = v - p[2 * w - 2]; d[15] = v - p[3 * w - 1];
    // cornerScore = (largest t such that 9 contiguous circle pixels are all > v + t or all < v - t), found by bisection on t with
    // 16-bit circle masks.  (A first version used min/max chains; ptxas fuses those into VIMNMX3 on sm_100a and the result came
    // out wrong on the B200 although the PTX was correct -- see profiles/r1_notes.md -- so this kernel avoids integer min/max.)
    auto is_corner = [&](int t) -> bool {
      unsigned br = 0, dk = 0;
#pragma unroll
      for (int k = 0; k < 16; ++k) { br |= (unsigned)(d[k] > t) << k; dk |= (unsigned)(d[k] < -t) << k; }
      auto nine = [](unsigned m) -> bool {
        m |= m << 16;                                   // unroll the circle
        unsigned a = m & (m >> 1);                      // 2 contiguous
        a &= a >> 2;                                    // 4
        a &= a >> 4;                                    // 8
        a &= m >> 8;                                    // 9
        return (a & 0xffffu) != 0u;
      };
      return nine(br) || nine(dk);
    };
    int lo = -1, hi = 255;                              // invariant: corner at lo (t = -1 is always true), not a corner at hi
#pragma unroll 1
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (is_corner(mid)) lo = mid; else hi = mid;
    }
    out = lo < 0 ? 0 : lo;
  }
  score[(size_t)y * w + x] = (unsigned char)out;
}

// ------------------------------------------------------------------------------------------------ per-cell FAST + NMS
struct Cell { int x0, y0, x1, y1, offx, offy; };   // ROI [x0,x1) x [y0,y1) in level coordinates; keypoint offset (j*wCell, i*hCell)
struct KpOut { float x, y, resp; };

// One CTA per cell.  Detection region = ROI minus a 3-px frame (cv::FAST on the ROI); NMS neighbours outside it count as 0;
// first threshold thr_hi, and if the cell stays empty thr_lo.  Output row-major, like cv::FAST.
__global__ void __launch_bounds__(256) k_fast_cells(const unsigned char* __restrict__ score, int w, const Cell* __restrict__ cells,
                                                    int thr_hi, int thr_lo, KpOut* __restrict__ out, int* __restrict__ count) {
  __shared__ unsigned char s[64 * 64];     // cell <= 60 px on a side (width / floor(width / 30) < 60) plus the zero halo
  __shared__ int wsum[8];
  __shared__ int total;
  const Cell c = cells[blockIdx.x];
  const int rx0 = c.x0 + 3, ry0 = c.y0 + 3, rw = c.x1 - c.x0 - 6, rh = c.y1 - c.y0 - 6;   // detection region
  const int pw = rw + 2, ph = rh + 2;                                                          // with a zero halo
  for (int i = threadIdx.x; i < pw * ph; i += blockDim.x) {
    const int lx = i % pw - 1, ly = i / pw - 1;
    s[i] = (lx >= 0 && ly >= 0 && lx < rw && ly < rh) ? score[(size_t)(ry0 + ly) * w + rx0 + lx] : 0;
  }
  __syncthreads();
  const int npx = rw * rh;
  const int per = (npx + blockDim.x - 1) / blockDim.x;        // contiguous row-major range per thread keeps the output ordered
  const int b = threadIdx.x * per, e = min(b + per, npx);
  for (int pass = 0; pass < 2; ++pass) {
    const int thr = pass == 0 ? thr_hi : thr_lo;
    int cnt = 0;
    for (int i = b; i < e; ++i) {
      const int lx = i % rw, ly = i / rw;
      const int v = s[(ly + 1) * pw + lx + 1];
      if (v < thr) continue;
      bool ismax = true;
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          if (dx == 0 && dy == 0) continue;
          int nb = s[(ly + 1 + dy) * pw + lx + 1 + dx];
          if (nb < thr) nb = 0;
          ismax = ismax && (v > nb);
        }
      cnt += ismax;
    }
    // exclusive scan of cnt over the CTA (warp shuffles + one smem hop)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) { int acc = 0; for (int k = 0; k < 8; ++k) { const int t = wsum[k]; wsum[k] = acc; acc += t; } total = acc; }
    __syncthreads();
    int pos = wsum[wid] + incl - cnt;
    const int tot = total;
    if (tot > 0) {
      KpOut* o = out + (size_t)blockIdx.x * CELL_CAP;
      for (int i = b; i < e; ++i) {
        const int lx = i % rw, ly = i / rw;
        const int v = s[(ly + 1) * pw + lx + 1];
        if (v < thr) continue;
        bool ismax = true;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx) {
            if (dx == 0 && dy == 0) continue;
            int nb = s[(ly + 1 + dy) * pw + lx + 1 + dx];
            if (nb < thr) nb = 0;
            ismax = ismax && (v > nb);
          }
        if (ismax) {
          if (pos < CELL_CAP) { o[pos].x = (float)(lx + 3 + c.offx); o[pos].y = (float)(ly + 3 + c.offy); o[pos].resp = (float)v; }
          ++pos;
        }
      }
      if (threadIdx.x == 0) count[blockIdx.x] = min(tot, CELL_CAP);
      return;                      // uniform: every thread sees the same `total`
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) count[blockIdx.x] = 0;
}

// ------------------------------------------------------------------------------------------------ IC_Angle
struct UmaxArg { int v[16]; };
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {   // cv::fastAtan2 (scalar path), no FMA contraction
  const float s = (float)(180.0 / 3.14159265358979323846);
  const float p1 = 0.9997878412794807f * s, p3 = -0.3258083974640975f * s, p5 = 0.1555786518463281f * s, p7 = -0.04432655554792128f * s;
  const float ax = fabsf(x), ay = fabsf(y), eps = 2.2204460492503131e-16f;
  float a, c, c2;
  if (ax >= ay) {
    c = __fdiv_rn(ay, __fadd_rn(ax, eps)); c2 = __fmul_rn(c, c);
    a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
  } else {
    c = __fdiv_rn(ax, __fadd_rn(ay, eps)); c2 = __fmul_rn(c, c);
    a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
  }
  if (x < 0) a = __fsub_rn(180.f, a);
  if (y < 0) a = __fsub_rn(360.f, a);
  return a;
}
struct KpLvl { float x, y; int level; };
struct LevelDesc { const unsigned char* img; int w, h; };
struct LevelsArg { LevelDesc L[MAX_LEVELS]; };
// one warp per keypoint: lanes stride over the rows v = 0..15 of the circular patch
__global__ void k_ic_angle(const KpLvl* __restrict__ kps, int n, float* __restrict__ angle, LevelsArg levels, UmaxArg umax) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n) return;
  const KpLvl k = kps[wid];
  const LevelDesc L = levels.L[k.level];
  const int cx = __float2int_rn(k.x), cy = __float2int_rn(k.y);
  int m01 = 0, m10 = 0;
  if (lane <= HALF_PATCH) {
    const int v = lane;
    if (v == 0) {
      const unsigned char* r = L.img + (size_t)cy * L.w + cx;
      for (int u = -HALF_PATCH; u <= HALF_PATCH; ++u) m10 += u * (int)r[u];
    } else {
      const int d = umax.v[v];
      const unsigned char* rp = L.img + (size_t)(cy + v) * L.w + cx;
      const unsigned char* rm = L.img + (size_t)(cy - v) * L.w + cx;
      int vs = 0;
      for (int u = -d; u <= d; ++u) { const int a = rp[u], b = rm[u]; vs += a - b; m10 += u * (a + b); }
      m01 = v * vs;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { m01 += __shfl_down_sync(0xffffffffu, m01, o); m10 += __shfl_down_sync(0xffffffffu, m10, o); }
  if (lane == 0) angle[wid] = fast_atan2_deg((float)m01, (float)m10);
}

// ------------------------------------------------------------------------------------------------ sampling (ordered compaction)
__device__ __forceinline__ int cta_excl_scan(int flag, int* wsum /*33*/, int& total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int incl = flag;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  __syncthreads();
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  if (threadIdx.x == 0) { int acc = 0; for (int k = 0; k < nw; ++k) { const int t = wsum[k]; wsum[k] = acc; acc += t; } wsum[32] = acc; }
  __syncthreads();
  total = wsum[32];
  return wsum[wid] + incl - flag;
}
struct ObjSample { int x, y; float cx, cy, fx, fy, depth; int label; };
// Frame.cc:200-228: stride-`step` raster scan, single CTA so that the output keeps the raster (push_back) order
__global__ void __launch_bounds__(1024) k_sample_objects(const int* __restrict__ mask, const float* __restrict__ depth, const float* __restrict__ flow,
                                                          int w, int h, int step, float th, ObjSample* __restrict__ out, int cap, int* __restrict__ n_out) {
  __shared__ int wsum[33];
  const int nx = (w + step - 1) / step, ny = (h + step - 1) / step, n = nx * ny;
  int base = 0;
  for (int start = 0; start < n; start += blockDim.x) {
    const int i = start + threadIdx.x;
    int ok = 0, x = 0, y = 0, m = 0; float d = 0, fx = 0, fy = 0, tx = 0, ty = 0;
    if (i < n) {
      x = (i % nx) * step; y = (i / nx) * step;
      const size_t p = (size_t)y * w + x;
      m = mask[p]; d = depth[p];
      if (m != 0 && d < th && d > 0.f) {
        fx = flow[2 * p]; fy = flow[2 * p + 1];
        tx = __fadd_rn((float)x, fx); ty = __fadd_rn((float)y, fy);
        ok = (tx < (float)w && tx > 0.f && ty < (float)h && ty > 0.f);
      }
    }
    int tot;
    const int pos = base + cta_excl_scan(ok, wsum, tot);
    if (ok && pos < cap) out[pos] = ObjSample{x, y, tx, ty, fx, fy, d, m};
    base += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_out = min(base, cap);
}
struct StatOut { int idx; float cx, cy, fu, fv, depth; };
// Frame.cc:100-129 + 181-194: keep ORB keypoints on static background with valid depth and non-zero flow staying in the image
__global__ void __launch_bounds__(1024) k_filter_static(const float* __restrict__ kx, const float* __restrict__ ky, int n, const int* __restrict__ mask,
                                                         const float* __restrict__ depth, const float* __restrict__ flow, int w, int h, float th,
                                                         StatOut* __restrict__ out, int* __restrict__ n_out) {
  __shared__ int wsum[33];
  int base = 0;
  for (int start = 0; start < n; start += blockDim.x) {
    const int i = start + threadIdx.x;
    int ok = 0; float fx = 0, fy = 0, px = 0, py = 0, dd = -1.f;
    if (i < n) {
      px = kx[i]; py = ky[i];
      const int x = (int)px, y = (int)py;
      const size_t p = (size_t)y * w + x;
      const float d = depth[p];
      if (mask[p] == 0 && !(d > th || d <= 0.f)) {
        fx = flow[2 * p]; fy = flow[2 * p + 1];
        if (fx != 0.f && fy != 0.f)
          ok = (__fadd_rn(px, fx) < (float)w && __fadd_rn(py, fy) < (float)h && px < (float)w && py < (float)h);
        if (ok) dd = d > 0.f ? d : -1.f;
      }
    }
    int tot;
    const int pos = base + cta_excl_scan(ok, wsum, tot);
    if (ok) out[pos] = StatOut{i, __fadd_rn(px, fx), __fadd_rn(py, fy), fx, fy, dd};
    base += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_out = base;
}

// ------------------------------------------------------------------------------------------------ sampled background keypoints
// Frame::SampleKeyPoints (src/Frame.cc:672-740) + Option II of the Frame constructor (:130-194).  cv::RNG is multiply-with-carry,
// s <- (s mod 2^32) * A + floor(s / 2^32), returning (uint32)s.  That step is s * r mod m with m = A * 2^32 - 1 and r = 2^-32 mod m
// (A * 2^32 == 1 mod m), so the state after k draws is seed * r^k mod m and every draw is independent of the others given a table
// of powers of r.  The reference's loop visits cell c = v % 400 at visit v (column cell i = c / 20 outer, row cell j = c % 20 inner)
// and draws x then y, i.e. draws 2v+1 and 2v+2.  Only the 39 cells with i == 0 or j == 0 can reject a visit, so 3 000 samples
// need at most 9 sweeps of 400 visits.
constexpr unsigned long long RNG_A = 4164903690ull, RNG_M = 0xf83f6309ffffffffull;
constexpr int SAMP_DIV = 20, SAMP_CELLS = SAMP_DIV * SAMP_DIV, SAMP_SWEEPS = 9, SAMP_VISITS = SAMP_CELLS * SAMP_SWEEPS, SAMP_DRAWS = 2 * SAMP_VISITS;
static_assert(VDO_SAMPLE_KEYPOINTS <= (SAMP_CELLS - 2 * SAMP_DIV + 1) * SAMP_SWEEPS, "9 sweeps must always yield the samples");

// (uint32)(seed * t * r^2 mod m) for seed < 2^32, t < m: two MWC steps on the 96-bit product (each multiplies by r), then one
// conditional subtraction (the second step leaves a value below m + 2^33 < 2m)
__device__ __forceinline__ unsigned rng_draw(unsigned seed, unsigned long long t) {
  const unsigned long long lo = (unsigned long long)seed * t, hi = __umul64hi((unsigned long long)seed, t);
  const unsigned long long a = (lo & 0xffffffffull) * RNG_A, s = a + ((hi << 32) | (lo >> 32));
  const unsigned long long carry = s < a;                                   // the first step can reach 2^65
  unsigned long long s2 = (s & 0xffffffffull) * RNG_A + ((carry << 32) | (s >> 32));
  if (s2 >= RNG_M) s2 -= RNG_M;
  return (unsigned)s2;
}
struct SampOut { float kx, ky, cx, cy, fu, fv, depth; };
// One CTA: the 3 000 kept visits depend on a prefix count over all visits, and their cell-major placement on counts over all cells.
// rpow[k] = r^(k-1) mod m, so draw k (1-based) is rng_draw(seed, rpow[k - 1]).
__global__ void __launch_bounds__(1024) k_sample_static(const unsigned long long* __restrict__ rpow, unsigned seed, const int* __restrict__ mask,
                                                         const float* __restrict__ depth, const float* __restrict__ flow, int w, int h, float th,
                                                         float* __restrict__ raw, SampOut* __restrict__ out, int* __restrict__ n_out) {
  __shared__ int vx[SAMP_VISITS], vy[SAMP_VISITS];
  __shared__ unsigned char keep[SAMP_VISITS];
  __shared__ short ord[VDO_SAMPLE_KEYPOINTS];           // visit of each output slot, cell-major
  __shared__ int wsum[33];
  const int xs = w / SAMP_DIV, ys = h / SAMP_DIV;
  // (1) draws and acceptance; the loop's `break` keeps the first VDO_SAMPLE_KEYPOINTS accepted visits
  int base = 0;
  for (int start = 0; start < SAMP_VISITS; start += blockDim.x) {
    const int v = start + threadIdx.x;
    int ok = 0;
    if (v < SAMP_VISITS) {
      const int c = v % SAMP_CELLS, i = c / SAMP_DIV, j = c % SAMP_DIV;
      const int x = i * xs + (int)(rng_draw(seed, rpow[2 * v]) % (unsigned)xs);        // rng.uniform(i*x_step, (i+1)*x_step)
      const int y = j * ys + (int)(rng_draw(seed, rpow[2 * v + 1]) % (unsigned)ys);
      ok = !(x >= w || y >= h || x <= 0 || y <= 0);
      vx[v] = x; vy[v] = y;
    }
    int tot;
    const int rank = base + cta_excl_scan(ok, wsum, tot);
    if (v < SAMP_VISITS) keep[v] = ok && rank < VDO_SAMPLE_KEYPOINTS;
    base += tot;
    __syncthreads();
  }
  // (2) cell-major placement (KeyinGrid[i*20+j] in draw order): slot = kept visits of the earlier cells + rank within the own cell
  int cnt = 0;
  if (threadIdx.x < SAMP_CELLS)
    for (int q = 0; q < SAMP_SWEEPS; ++q) cnt += keep[threadIdx.x + q * SAMP_CELLS];
  int n_raw;
  int pos = cta_excl_scan(cnt, wsum, n_raw);
  if (threadIdx.x < SAMP_CELLS)
    for (int q = 0; q < SAMP_SWEEPS; ++q) {
      const int v = threadIdx.x + q * SAMP_CELLS;
      if (keep[v]) ord[pos++] = (short)v;
    }
  __syncthreads();
  if (raw)
    for (int k = threadIdx.x; k < n_raw; k += blockDim.x) { raw[2 * k] = (float)vx[ord[k]]; raw[2 * k + 1] = (float)vy[ord[k]]; }
  // (3) Option II filter, ordered compaction
  base = 0;
  for (int start = 0; start < n_raw; start += blockDim.x) {
    const int k = start + threadIdx.x;
    int ok = 0; float px = 0, py = 0, fx = 0, fy = 0, tx = 0, ty = 0, d = 0;
    if (k < n_raw) {
      const int x = vx[ord[k]], y = vy[ord[k]];
      px = (float)x; py = (float)y;
      const size_t p = (size_t)y * w + x;
      d = depth[p];
      if (mask[p] == 0 && !(d > th || d <= 0.f)) {
        fx = flow[2 * p]; fy = flow[2 * p + 1];
        if (fx != 0.f && fy != 0.f) {
          tx = __fadd_rn(px, fx); ty = __fadd_rn(py, fy);
          ok = (tx < (float)w && ty < (float)h && tx > 0.f && ty > 0.f);
        }
      }
    }
    int tot;
    const int o = base + cta_excl_scan(ok, wsum, tot);
    if (ok) out[o] = SampOut{px, py, tx, ty, fx, fy, d > 0.f ? d : -1.f};
    base += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_out = base;
}

// Dense packing of the per-cell candidate lists (cell-major, row-major inside a cell = the order the host octree expects):
// k_cell_offsets: exclusive scan of the cell counts by one CTA; k_cell_gather: one CTA per cell copies its entries.
// Only count + offsets (a few KB) and the packed candidates (~0.3 MB) cross PCIe instead of ncell * CELL_CAP slots (~8 MB).
__global__ void __launch_bounds__(1024) k_cell_offsets(const int* __restrict__ count, int n, int* __restrict__ offset) {
  __shared__ int s[1024];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < n ? count[i] : 0;
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const int t = threadIdx.x >= o ? s[threadIdx.x - o] : 0;
      __syncthreads();
      s[threadIdx.x] += t;
      __syncthreads();
    }
    if (i < n) offset[i] = carry + s[threadIdx.x] - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry += s[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) offset[n] = carry;
}
__global__ void k_cell_gather(const KpOut* __restrict__ cell_out, const int* __restrict__ count, const int* __restrict__ offset, KpOut* __restrict__ dense) {
  const int c = blockIdx.x, n = count[c], o = offset[c];
  for (int k = threadIdx.x; k < n; k += blockDim.x) dense[o + k] = cell_out[(size_t)c * CELL_CAP + k];
}

// ------------------------------------------------------------------------------------------------ back-projection / scene flow
struct Pose32 { float R[9], t[3]; };   // Tcw rows
// X_w = Rwl * x3Dc + twl as a cv::Mat float gemm: products accumulated in double, one rounding to float (twl itself is float)
__device__ __forceinline__ void unproject_world(float u, float v, float z, const float* K, const Pose32& T, float* X) {
  const float invfx = __fdiv_rn(1.f, K[0]), invfy = __fdiv_rn(1.f, K[1]);
  const float x = __fmul_rn(__fmul_rn(__fsub_rn(u, K[2]), z), invfx), y = __fmul_rn(__fmul_rn(__fsub_rn(v, K[3]), z), invfy);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double twl = (double)(float)(-((double)T.R[r] * (double)T.t[0] + (double)T.R[3 + r] * (double)T.t[1] + (double)T.R[6 + r] * (double)T.t[2]));
    X[r] = (float)((double)T.R[r] * (double)x + (double)T.R[3 + r] * (double)y + (double)T.R[6 + r] * (double)z + twl);
  }
}
__global__ void k_scene_flow(int n, const float* __restrict__ up, const float* __restrict__ vp, const float* __restrict__ zp, Pose32 Tp,
                             const float* __restrict__ uc, const float* __restrict__ vc, const float* __restrict__ zc, Pose32 Tc,
                             const int* __restrict__ labp, const int* __restrict__ labc, float4 K, float* __restrict__ flow3d,
                             float* __restrict__ Xp_out, unsigned char* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float Kf[4] = {K.x, K.y, K.z, K.w};
  float Xp[3], Xc[3];
  unproject_world(up[i], vp[i], zp[i], Kf, Tp, Xp);
  unproject_world(uc[i], vc[i], zc[i], Kf, Tc, Xc);
  const bool ok = labc[i] > 0 && labp[i] > 0;
  valid[i] = ok;
#pragma unroll
  for (int r = 0; r < 3; ++r) { flow3d[3 * i + r] = ok ? __fsub_rn(Xc[r], Xp[r]) : 0.f; if (Xp_out) Xp_out[3 * i + r] = Xp[r]; }
}

// ------------------------------------------------------------------------------------------------ host side
struct OrbSetup {
  int nfeatures = 0, nlevels = 0, ini_th = 0, min_th = 0;
  float scale_factor[MAX_LEVELS], inv_scale[MAX_LEVELS];
  int per_level[MAX_LEVELS];
  int umax[16];
  void init(int nf, float sf, int nl, int ini, int mn) {
    nfeatures = nf; nlevels = nl; ini_th = ini; min_th = mn;
    scale_factor[0] = 1.f;
    for (int i = 1; i < nl; ++i) scale_factor[i] = scale_factor[i - 1] * sf;
    for (int i = 0; i < nl; ++i) inv_scale[i] = 1.f / scale_factor[i];
    float factor = 1.f / sf;
    float nd = nf * (1 - factor) / (1 - (float)std::pow((double)factor, (double)nl));
    int sum = 0;
    for (int l = 0; l < nl - 1; ++l) { per_level[l] = (int)std::lrint(nd); sum += per_level[l]; nd *= factor; }
    per_level[nl - 1] = std::max(nf - sum, 0);
    int vmax = (int)std::floor(HALF_PATCH * std::sqrt(2.f) / 2 + 1), vmin = (int)std::ceil(HALF_PATCH * std::sqrt(2.f) / 2);
    const double hp2 = HALF_PATCH * HALF_PATCH;
    for (int v = 0; v <= vmax; ++v) umax[v] = (int)std::lrint(std::sqrt(hp2 - v * v));
    for (int v = HALF_PATCH, v0 = 0; v >= vmin; --v) { while (umax[v0] == umax[v0 + 1]) ++v0; umax[v] = v0; ++v0; }
  }
};

// ---- DistributeOctTree (src/ORBextractor.cc:470-752) on the host: a serial, order-dependent procedure over a few thousand
// candidates.  Tie rule for equally sized nodes: the later-created node is expanded first (the reference compares heap pointers).
struct OKey { float x, y, r; };
struct ONode {
  int ULx, ULy, URx, URy, BLx, BLy, BRx, BRy;
  std::vector<OKey> keys;
  bool no_more = false;
  long seq = 0;
  std::list<ONode>::iterator lit;
};
static void divide_node(const ONode& n, ONode c[4]) {
  const int halfX = (int)std::ceil(static_cast<float>(n.URx - n.ULx) / 2), halfY = (int)std::ceil(static_cast<float>(n.BRy - n.ULy) / 2);
  c[0].ULx = n.ULx; c[0].ULy = n.ULy; c[0].URx = n.ULx + halfX; c[0].URy = n.ULy; c[0].BLx = n.ULx; c[0].BLy = n.ULy + halfY; c[0].BRx = n.ULx + halfX; c[0].BRy = n.ULy + halfY;
  c[1].ULx = c[0].URx; c[1].ULy = c[0].URy; c[1].URx = n.URx; c[1].URy = n.URy; c[1].BLx = c[0].BRx; c[1].BLy = c[0].BRy; c[1].BRx = n.URx; c[1].BRy = n.ULy + halfY;
  c[2].ULx = c[0].BLx; c[2].ULy = c[0].BLy; c[2].URx = c[0].BRx; c[2].URy = c[0].BRy; c[2].BLx = n.BLx; c[2].BLy = n.BLy; c[2].BRx = c[0].BRx; c[2].BRy = n.BLy;
  c[3].ULx = c[2].URx; c[3].ULy = c[2].URy; c[3].URx = c[1].BRx; c[3].URy = c[1].BRy; c[3].BLx = c[2].BRx; c[3].BLy = c[2].BRy; c[3].BRx = n.BRx; c[3].BRy = n.BRy;
  for (const OKey& k : n.keys) {
    if (k.x < c[0].URx) { if (k.y < c[0].BRy) c[0].keys.push_back(k); else c[2].keys.push_back(k); }
    else if (k.y < c[0].BRy) c[1].keys.push_back(k);
    else c[3].keys.push_back(k);
  }
  for (int i = 0; i < 4; ++i) if (c[i].keys.size() == 1) c[i].no_more = true;
}
static std::vector<OKey> distribute_octtree(const std::vector<OKey>& in, int minX, int maxX, int minY, int maxY, int N) {
  std::vector<OKey> res;
  if (in.empty()) return res;
  const int nIni = (int)std::round(static_cast<float>(maxX - minX) / (maxY - minY));
  const float hX = static_cast<float>(maxX - minX) / nIni;
  std::list<ONode> nodes;
  std::vector<ONode*> ini(nIni);
  long seq = 0;
  for (int i = 0; i < nIni; ++i) {
    ONode n;
    n.ULx = (int)(hX * static_cast<float>(i)); n.ULy = 0; n.URx = (int)(hX * static_cast<float>(i + 1)); n.URy = 0;
    n.BLx = n.ULx; n.BLy = maxY - minY; n.BRx = n.URx; n.BRy = maxY - minY;
    nodes.push_back(n); ini[i] = &nodes.back();
  }
  for (const OKey& k : in) ini[(int)(k.x / hX)]->keys.push_back(k);
  for (auto it = nodes.begin(); it != nodes.end();) {
    if (it->keys.size() == 1) { it->no_more = true; ++it; }
    else if (it->keys.empty()) it = nodes.erase(it);
    else ++it;
  }
  auto push_children = [&](const ONode& parent, std::vector<ONode*>& expand) {
    ONode c[4];
    divide_node(parent, c);
    for (int i = 0; i < 4; ++i)
      if (!c[i].keys.empty()) {
        c[i].seq = ++seq;
        nodes.push_front(c[i]);
        nodes.front().lit = nodes.begin();
        if (nodes.front().keys.size() > 1) expand.push_back(&nodes.front());
      }
  };
  bool finish = false;
  std::vector<ONode*> expand;
  while (!finish) {
    const int prev = (int)nodes.size();
    expand.clear();
    for (auto it = nodes.begin(); it != nodes.end();) {
      if (it->no_more) { ++it; continue; }
      push_children(*it, expand);
      it = nodes.erase(it);
    }
    if ((int)nodes.size() >= N || (int)nodes.size() == prev) finish = true;
    else if ((int)nodes.size() + (int)expand.size() * 3 > N) {
      while (!finish) {
        const int prev2 = (int)nodes.size();
        std::vector<ONode*> pe = expand;
        expand.clear();
        std::sort(pe.begin(), pe.end(), [](const ONode* a, const ONode* b) { return a->keys.size() != b->keys.size() ? a->keys.size() < b->keys.size() : a->seq < b->seq; });
        for (int j = (int)pe.size() - 1; j >= 0; --j) {
          push_children(*pe[j], expand);
          nodes.erase(pe[j]->lit);
          if ((int)nodes.size() >= N) break;
        }
        if ((int)nodes.size() >= N || (int)nodes.size() == prev2) finish = true;
      }
    }
  }
  res.reserve(nodes.size());
  for (const ONode& n : nodes) {
    const OKey* best = &n.keys[0];
    for (size_t k = 1; k < n.keys.size(); ++k) if (n.keys[k].r > best->r) best = &n.keys[k];
    res.push_back(*best);
  }
  return res;
}

}  // namespace

// ================================================================================================ C ABI

// ------------------------------------------------------------------------------------------------ descriptors (A6)
// GaussianBlur(level, Size(7,7), 2, 2, BORDER_REFLECT_101) as OpenCV computes it for CV_8U (fixed point, bit-exact against cv2 4.13):
// Q8.8 kernel {18, 34, 48, 56, 48, 34, 18} / 256, horizontal pass kept in Q8.8, vertical pass in Q16.16, (v + 2^15) >> 16.
// (src/ORBextractor.cc:1083-1084.  OpenCV 3.4.0, which the reference's Dockerfile builds, still filtered in float: version drift.)
__device__ __forceinline__ int reflect101(int p, int n) { if (p < 0) p = -p; if (p >= n) p = 2 * n - 2 - p; return p; }
__global__ void k_blur7(const unsigned char* __restrict__ src, int w, int h, unsigned char* __restrict__ dst) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const int kq[7] = {18, 34, 48, 56, 48, 34, 18};
  int xs[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) xs[i] = reflect101(x + i - 3, w);
  unsigned int v = 0;
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const unsigned char* row = src + (size_t)reflect101(y + j - 3, h) * w;
    unsigned int hsum = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i) hsum += (unsigned int)kq[i] * row[xs[i]];
    v += (unsigned int)kq[j] * hsum;
  }
  dst[(size_t)y * w + x] = (unsigned char)((v + (1u << 15)) >> 16);
}
// computeOrbDescriptor (src/ORBextractor.cc:97-136): one warp per keypoint, one descriptor byte (8 pair tests) per lane.
__constant__ signed char c_orb_pattern[1024] = {
#include "orb_pattern.inc"
};
struct BlurLevels { const unsigned char* img[MAX_LEVELS]; int w[MAX_LEVELS], h[MAX_LEVELS]; };
__global__ void k_orb_descriptors(const KpLvl* __restrict__ kps, const float* __restrict__ ang, int n, BlurLevels L, unsigned char* __restrict__ desc) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= n) return;
  const KpLvl kp = kps[k];
  const float factorPI = (float)(3.14159265358979323846 / 180.f);
  const float angle = __fmul_rn(ang[k], factorPI);
  const float a = (float)cos((double)angle), b = (float)sin((double)angle);
  const int w = L.w[kp.level];
  const unsigned char* center = L.img[kp.level] + (size_t)__float2int_rn(kp.y) * w + __float2int_rn(kp.x);
  int val = 0;
#pragma unroll
  for (int bit = 0; bit < 8; ++bit) {
    const signed char* pt = c_orb_pattern + 4 * (8 * lane + bit);
    int t[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const float px = (float)pt[2 * q], py = (float)pt[2 * q + 1];
      const int iy = __float2int_rn(__fadd_rn(__fmul_rn(px, b), __fmul_rn(py, a)));
      const int ix = __float2int_rn(__fsub_rn(__fmul_rn(px, a), __fmul_rn(py, b)));
      t[q] = center[iy * w + ix];
    }
    val |= (t[0] < t[1]) << bit;
  }
  desc[(size_t)k * 32 + lane] = (unsigned char)val;
}

struct vdo_frame {
  vdo_ctx* ctx; cudaStream_t st;
  int w, h;
  unsigned char* gray = nullptr; float* depth = nullptr; float* flow = nullptr; int* mask = nullptr;
  unsigned char* pyr[MAX_LEVELS] = {nullptr}; unsigned char* score[MAX_LEVELS] = {nullptr}; int lw[MAX_LEVELS], lh[MAX_LEVELS];
  Cell* cells = nullptr; KpOut* cell_out = nullptr; int* cell_cnt = nullptr; int cells_cap = 0;
  int* cell_off = nullptr; KpOut* cell_dense = nullptr; int* h_cnt_off = nullptr; KpOut* h_dense = nullptr; size_t h_dense_cap = 0;   // packed candidates (pinned host side)
  KpLvl* kps = nullptr; float* ang = nullptr; int kp_cap = 0, n_kps = -1;    // keypoints (level coordinates) / angles of the last vdo_orb_extract
  unsigned char* blur[MAX_LEVELS] = {nullptr};
  void* scratch = nullptr; size_t scratch_cap = 0; int* d_count = nullptr;
  unsigned long long* samp_pow = nullptr;        // r^(k-1) mod m for the SAMP_DRAWS draws of vdo_frame_sample_static (seed-independent)
  std::vector<KpOut> h_cell_out; std::vector<int> h_cell_cnt;
  OrbSetup orb; bool orb_ready = false;
  int launches = 0;
};

static int ensure_scratch(vdo_frame* f, size_t bytes) {
  if (bytes <= f->scratch_cap) return VDO_OK;
  cudaFree(f->scratch);
  FRK(cudaMalloc(&f->scratch, bytes * 2));
  f->scratch_cap = bytes * 2;
  return VDO_OK;
}

extern "C" int vdo_frame_create(vdo_ctx* ctx, int width, int height, vdo_frame** out) {
  if (!ctx || !out || width < 64 || height < 64) return VDO_ERR_ARG;
  vdo_frame* f = new vdo_frame;
  f->ctx = ctx; f->st = (cudaStream_t)(uintptr_t)vdo_ctx_stream(ctx); f->w = width; f->h = height;
  const size_t n = (size_t)width * height;
  FRK(cudaMalloc(&f->gray, n)); FRK(cudaMalloc(&f->depth, n * 4)); FRK(cudaMalloc(&f->flow, n * 8)); FRK(cudaMalloc(&f->mask, n * 4));
  FRK(cudaMalloc(&f->d_count, 64));
  *out = f;
  return VDO_OK;
}
extern "C" void vdo_frame_destroy(vdo_frame* f) {
  if (!f) return;
  cudaFree(f->gray); cudaFree(f->depth); cudaFree(f->flow); cudaFree(f->mask); cudaFree(f->d_count);
  for (int l = 1; l < MAX_LEVELS; ++l) cudaFree(f->pyr[l]);
  for (int l = 0; l < MAX_LEVELS; ++l) { cudaFree(f->score[l]); cudaFree(f->blur[l]); }
  cudaFree(f->cells); cudaFree(f->cell_out); cudaFree(f->cell_cnt); cudaFree(f->kps); cudaFree(f->ang); cudaFree(f->scratch);
  cudaFree(f->cell_off); cudaFree(f->cell_dense); cudaFreeHost(f->h_cnt_off); cudaFreeHost(f->h_dense); cudaFree(f->samp_pow);
  delete f;
}
// D2H of the resident mask (the tracker writes it back into the caller's buffer only when UpdateMask changed it)
extern "C" int vdo_frame_read_mask(vdo_frame* f, int* mask_out) {
  if (!f || !mask_out) return VDO_ERR_ARG;
  FRK(cudaMemcpyAsync(mask_out, f->mask, sizeof(int) * (size_t)f->w * f->h, cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  return VDO_OK;
}
// internal: device pointers of a resident frame for the other translation units (tracking_ops.cu)
extern "C" int vdo_frame_device_ptrs(vdo_frame* f, unsigned char** gray, float** depth, float** flow, int** mask, int* w, int* h, void** stream) {
  if (!f) return VDO_ERR_ARG;
  if (gray) *gray = f->gray; if (depth) *depth = f->depth; if (flow) *flow = f->flow; if (mask) *mask = f->mask;
  if (w) *w = f->w; if (h) *h = f->h; if (stream) *stream = (void*)f->st;
  return VDO_OK;
}
// any of the four pointers may be NULL (keep what is resident)
extern "C" int vdo_frame_upload(vdo_frame* f, const unsigned char* gray, const float* depth, const float* flow, const int* mask) {
  if (!f) return VDO_ERR_ARG;
  const size_t n = (size_t)f->w * f->h;
  if (gray) FRK(cudaMemcpyAsync(f->gray, gray, n, cudaMemcpyHostToDevice, f->st));
  if (depth) FRK(cudaMemcpyAsync(f->depth, depth, n * 4, cudaMemcpyHostToDevice, f->st));
  if (flow) FRK(cudaMemcpyAsync(f->flow, flow, n * 8, cudaMemcpyHostToDevice, f->st));
  if (mask) FRK(cudaMemcpyAsync(f->mask, mask, n * 4, cudaMemcpyHostToDevice, f->st));
  return VDO_OK;
}
extern "C" int vdo_frame_depth_prep(vdo_frame* f, float bf, float factor, float* depth_out) {
  if (!f) return VDO_ERR_ARG;
  const int n = f->w * f->h;
  k_depth_prep<<<(n + 255) / 256, 256, 0, f->st>>>(f->depth, n, bf, factor); f->launches++;
  if (depth_out) { FRK(cudaMemcpyAsync(depth_out, f->depth, (size_t)n * 4, cudaMemcpyDeviceToHost, f->st)); FRK(cudaStreamSynchronize(f->st)); }
  return VDO_OK;
}

extern "C" int vdo_orb_extract(vdo_frame* f, int nfeatures, float scale_factor, int nlevels, int ini_th, int min_th, int max_out,
                               float* x, float* y, int* octave, float* response, float* angle, int* size, int* n_out, int* n_candidates) {
  if (!f || nlevels < 1 || nlevels > MAX_LEVELS || !x || !y || !n_out) return VDO_ERR_ARG;
  if (!f->orb_ready || f->orb.nfeatures != nfeatures || f->orb.nlevels != nlevels || f->orb.ini_th != ini_th || f->orb.min_th != min_th) {
    f->orb.init(nfeatures, scale_factor, nlevels, ini_th, min_th);
    f->orb_ready = true;
  }
  const OrbSetup& P = f->orb;
  // ---- pyramid + score maps ----
  f->pyr[0] = f->gray; f->lw[0] = f->w; f->lh[0] = f->h;
  LevelsArg lva; std::memset(&lva, 0, sizeof lva);
  LevelDesc* lv = lva.L;
  for (int l = 0; l < nlevels; ++l) {
    if (l > 0) {
      f->lw[l] = (int)std::lrint((float)f->w * P.inv_scale[l]); f->lh[l] = (int)std::lrint((float)f->h * P.inv_scale[l]);
      if (!f->pyr[l]) FRK(cudaMalloc(&f->pyr[l], (size_t)f->lw[l] * f->lh[l]));
      dim3 b(32, 8), g((f->lw[l] + 31) / 32, (f->lh[l] + 7) / 8);
      k_resize_u8<<<g, b, 0, f->st>>>(f->pyr[l - 1], f->lw[l - 1], f->lh[l - 1], f->pyr[l], f->lw[l], f->lh[l]); f->launches++;
    }
    if (!f->score[l]) FRK(cudaMalloc(&f->score[l], (size_t)f->lw[l] * f->lh[l]));
    dim3 b(32, 8), g((f->lw[l] + 31) / 32, (f->lh[l] + 7) / 8);
    k_fast_score<<<g, b, 0, f->st>>>(f->pyr[l], f->lw[l], f->lh[l], f->score[l]); f->launches++;
    lv[l] = LevelDesc{f->pyr[l], f->lw[l], f->lh[l]};
  }
  // ---- cell grids of all levels (ComputeKeyPointsOctTree geometry) ----
  std::vector<Cell> cells; std::vector<int> cell_begin(nlevels + 1, 0);
  int bord[MAX_LEVELS][4];
  for (int l = 0; l < nlevels; ++l) {
    const int minB = EDGE_THRESHOLD - 3, maxBX = f->lw[l] - EDGE_THRESHOLD + 3, maxBY = f->lh[l] - EDGE_THRESHOLD + 3;
    bord[l][0] = minB; bord[l][1] = maxBX; bord[l][2] = minB; bord[l][3] = maxBY;
    const float width = (float)(maxBX - minB), height = (float)(maxBY - minB);
    const int nCols = (int)(width / 30.f), nRows = (int)(height / 30.f);
    if (nCols < 1 || nRows < 1) { cell_begin[l + 1] = (int)cells.size(); continue; }
    const int wCell = (int)std::ceil(width / nCols), hCell = (int)std::ceil(height / nRows);
    if (wCell + 2 > 64 || hCell + 2 > 64) return VDO_ERR_UNSUPPORTED;
    for (int i = 0; i < nRows; ++i) {
      const int iniY = minB + i * hCell; int maxY = iniY + hCell + 6;
      if (iniY >= maxBY - 3) continue;
      if (maxY > maxBY) maxY = maxBY;
      for (int j = 0; j < nCols; ++j) {
        const int iniX = minB + j * wCell; int maxX = iniX + wCell + 6;
        if (iniX >= maxBX - 6) continue;
        if (maxX > maxBX) maxX = maxBX;
        cells.push_back(Cell{iniX, iniY, maxX, maxY, j * wCell, i * hCell});
      }
    }
    cell_begin[l + 1] = (int)cells.size();
  }
  const int ncell = (int)cells.size();
  if (ncell > f->cells_cap) {
    cudaFree(f->cells); cudaFree(f->cell_out); cudaFree(f->cell_cnt);
    FRK(cudaMalloc(&f->cells, sizeof(Cell) * ncell)); FRK(cudaMalloc(&f->cell_out, sizeof(KpOut) * (size_t)ncell * CELL_CAP)); FRK(cudaMalloc(&f->cell_cnt, sizeof(int) * ncell));
    f->cells_cap = ncell; f->h_cell_cnt.resize(ncell);
    cudaFree(f->cell_off); cudaFree(f->cell_dense); cudaFreeHost(f->h_cnt_off);
    FRK(cudaMalloc(&f->cell_off, sizeof(int) * (ncell + 1))); FRK(cudaMalloc(&f->cell_dense, sizeof(KpOut) * (size_t)ncell * CELL_CAP));
    FRK(cudaMallocHost(&f->h_cnt_off, sizeof(int) * (2 * ncell + 1)));
  }
  FRK(cudaMemcpyAsync(f->cells, cells.data(), sizeof(Cell) * ncell, cudaMemcpyHostToDevice, f->st));
  for (int l = 0; l < nlevels; ++l) {
    const int nc = cell_begin[l + 1] - cell_begin[l];
    if (nc <= 0) continue;
    k_fast_cells<<<nc, 256, 0, f->st>>>(f->score[l], f->lw[l], f->cells + cell_begin[l], ini_th, min_th, f->cell_out + (size_t)cell_begin[l] * CELL_CAP, f->cell_cnt + cell_begin[l]);
    f->launches++;
  }
  k_cell_offsets<<<1, 1024, 0, f->st>>>(f->cell_cnt, ncell, f->cell_off); f->launches++;
  k_cell_gather<<<ncell, 64, 0, f->st>>>(f->cell_out, f->cell_cnt, f->cell_off, f->cell_dense); f->launches++;
  FRK(cudaMemcpyAsync(f->h_cnt_off, f->cell_cnt, sizeof(int) * ncell, cudaMemcpyDeviceToHost, f->st));
  FRK(cudaMemcpyAsync(f->h_cnt_off + ncell, f->cell_off, sizeof(int) * (ncell + 1), cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  const int* h_cnt = f->h_cnt_off; const int* h_off = f->h_cnt_off + ncell;
  const size_t n_dense = (size_t)h_off[ncell];
  if (n_dense > f->h_dense_cap) { cudaFreeHost(f->h_dense); FRK(cudaMallocHost(&f->h_dense, sizeof(KpOut) * n_dense * 2)); f->h_dense_cap = n_dense * 2; }
  if (n_dense) { FRK(cudaMemcpyAsync(f->h_dense, f->cell_dense, sizeof(KpOut) * n_dense, cudaMemcpyDeviceToHost, f->st)); FRK(cudaStreamSynchronize(f->st)); }
  // ---- octree distribution per level (host) ----
  std::vector<KpLvl> sel; std::vector<float> resp; std::vector<int> lvl_of;
  for (int l = 0; l < nlevels; ++l) {
    std::vector<OKey> cand;
    for (int c = cell_begin[l]; c < cell_begin[l + 1]; ++c)
      for (int k = 0; k < h_cnt[c]; ++k) { const KpOut& o = f->h_dense[(size_t)h_off[c] + k]; cand.push_back(OKey{o.x, o.y, o.resp}); }
    if (n_candidates) n_candidates[l] = (int)cand.size();
    std::vector<OKey> kept = distribute_octtree(cand, bord[l][0], bord[l][1], bord[l][2], bord[l][3], P.per_level[l]);
    for (const OKey& k : kept) { sel.push_back(KpLvl{k.x + (float)bord[l][0], k.y + (float)bord[l][2], l}); resp.push_back(k.r); }
  }
  const int n = (int)sel.size();
  *n_out = std::min(n, max_out);
  f->n_kps = angle ? n : -1;
  if (n == 0) return VDO_OK;
  if (n > f->kp_cap) { cudaFree(f->kps); cudaFree(f->ang); FRK(cudaMalloc(&f->kps, sizeof(KpLvl) * n * 2)); FRK(cudaMalloc(&f->ang, sizeof(float) * n * 2)); f->kp_cap = n * 2; }
  std::vector<float> h_ang(n, -1.f);
  if (angle) {
    FRK(cudaMemcpyAsync(f->kps, sel.data(), sizeof(KpLvl) * n, cudaMemcpyHostToDevice, f->st));
    UmaxArg ua; for (int i = 0; i < 16; ++i) ua.v[i] = P.umax[i];
    k_ic_angle<<<(n * 32 + 255) / 256, 256, 0, f->st>>>(f->kps, n, f->ang, lva, ua); f->launches++;
    FRK(cudaMemcpyAsync(h_ang.data(), f->ang, sizeof(float) * n, cudaMemcpyDeviceToHost, f->st));
    FRK(cudaStreamSynchronize(f->st));
  }
  for (int i = 0; i < *n_out; ++i) {
    const int l = sel[i].level;
    float px = sel[i].x, py = sel[i].y;
    if (l != 0) { px *= P.scale_factor[l]; py *= P.scale_factor[l]; }
    x[i] = px; y[i] = py;
    if (octave) octave[i] = l;
    if (response) response[i] = resp[i];
    if (angle) angle[i] = h_ang[i];
    if (size) size[i] = (int)(PATCH_SIZE * P.scale_factor[l]);
  }
  return VDO_OK;
}

// Descriptors of the keypoints of the last vdo_orb_extract call (which must have asked for angles): 7x7 sigma-2 blur of every level that has
// keypoints, then the 256 rotated pair tests.  desc_out: n x 32 bytes, in the order vdo_orb_extract returned the keypoints.
extern "C" int vdo_orb_describe(vdo_frame* f, int n, unsigned char* desc_out) {
  if (!f || !f->orb_ready || n < 0 || (n && !desc_out)) return VDO_ERR_ARG;
  if (f->n_kps < 0 || n > f->n_kps) return VDO_ERR_STATE;
  if (n == 0) return VDO_OK;
  BlurLevels L; std::memset(&L, 0, sizeof L);
  for (int l = 0; l < f->orb.nlevels; ++l) {
    if (!f->blur[l]) FRK(cudaMalloc(&f->blur[l], (size_t)f->lw[l] * f->lh[l]));
    dim3 b(32, 8), g((f->lw[l] + 31) / 32, (f->lh[l] + 7) / 8);
    k_blur7<<<g, b, 0, f->st>>>(f->pyr[l], f->lw[l], f->lh[l], f->blur[l]); f->launches++;
    L.img[l] = f->blur[l]; L.w[l] = f->lw[l]; L.h[l] = f->lh[l];
  }
  if (int rc = ensure_scratch(f, (size_t)n * 32 + 64)) return rc;
  unsigned char* d_desc = (unsigned char*)f->scratch;
  k_orb_descriptors<<<(n * 32 + 255) / 256, 256, 0, f->st>>>(f->kps, f->ang, n, L, d_desc); f->launches++;
  FRK(cudaMemcpyAsync(desc_out, d_desc, (size_t)n * 32, cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  return VDO_OK;
}
// test hook: the blurred level of the last vdo_orb_describe call
extern "C" int vdo_frame_debug_blur(vdo_frame* f, int level, unsigned char* img_out) {
  if (!f || !f->orb_ready || level < 0 || level >= f->orb.nlevels || !f->blur[level] || !img_out) return VDO_ERR_ARG;
  FRK(cudaMemcpyAsync(img_out, f->blur[level], (size_t)f->lw[level] * f->lh[level], cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  return VDO_OK;
}

extern "C" int vdo_frame_sample_objects(vdo_frame* f, float th_depth_obj, int step, int max_out, int* x, int* y, float* cx, float* cy,
                                        float* fx, float* fy, float* depth, int* label, int* n_out) {
  if (!f || step < 1 || max_out < 0 || !n_out) return VDO_ERR_ARG;
  if (int rc = ensure_scratch(f, sizeof(ObjSample) * (size_t)max_out + 64)) return rc;
  ObjSample* d_out = (ObjSample*)f->scratch;
  k_sample_objects<<<1, 1024, 0, f->st>>>(f->mask, f->depth, f->flow, f->w, f->h, step, th_depth_obj, d_out, max_out, f->d_count); f->launches++;
  int n = 0;
  FRK(cudaMemcpyAsync(&n, f->d_count, sizeof(int), cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  std::vector<ObjSample> h(n);
  if (n) { FRK(cudaMemcpyAsync(h.data(), d_out, sizeof(ObjSample) * n, cudaMemcpyDeviceToHost, f->st)); FRK(cudaStreamSynchronize(f->st)); }
  for (int i = 0; i < n; ++i) { x[i] = h[i].x; y[i] = h[i].y; cx[i] = h[i].cx; cy[i] = h[i].cy; fx[i] = h[i].fx; fy[i] = h[i].fy; depth[i] = h[i].depth; label[i] = h[i].label; }
  *n_out = n;
  return VDO_OK;
}

extern "C" int vdo_frame_filter_static(vdo_frame* f, int n, const float* kx, const float* ky, float th_depth, int* keep_idx, float* cx, float* cy,
                                       float* fu, float* fv, float* depth, int* n_out) {
  if (!f || n < 0 || !n_out) return VDO_ERR_ARG;
  if (n == 0) { *n_out = 0; return VDO_OK; }
  const size_t need = sizeof(float) * 2 * (size_t)n + sizeof(StatOut) * (size_t)n + 64;
  if (int rc = ensure_scratch(f, need)) return rc;
  float* d_kx = (float*)f->scratch; float* d_ky = d_kx + n; StatOut* d_out = (StatOut*)(d_ky + n);
  FRK(cudaMemcpyAsync(d_kx, kx, sizeof(float) * n, cudaMemcpyHostToDevice, f->st));
  FRK(cudaMemcpyAsync(d_ky, ky, sizeof(float) * n, cudaMemcpyHostToDevice, f->st));
  k_filter_static<<<1, 1024, 0, f->st>>>(d_kx, d_ky, n, f->mask, f->depth, f->flow, f->w, f->h, th_depth, d_out, f->d_count); f->launches++;
  int m = 0;
  FRK(cudaMemcpyAsync(&m, f->d_count, sizeof(int), cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  std::vector<StatOut> h(m);
  if (m) { FRK(cudaMemcpyAsync(h.data(), d_out, sizeof(StatOut) * m, cudaMemcpyDeviceToHost, f->st)); FRK(cudaStreamSynchronize(f->st)); }
  for (int i = 0; i < m; ++i) { keep_idx[i] = h[i].idx; cx[i] = h[i].cx; cy[i] = h[i].cy; fu[i] = h[i].fu; fv[i] = h[i].fv; depth[i] = h[i].depth; }
  *n_out = m;
  return VDO_OK;
}

extern "C" int vdo_frame_sample_static(vdo_frame* f, uint32_t seed, float th_depth, int max_out, float* kx, float* ky, float* cx, float* cy, float* fu,
                                       float* fv, float* depth, int* n_out, float* raw_xy) {
  if (!f || max_out < 0 || !n_out || (max_out && (!kx || !ky || !cx || !cy || !fu || !fv || !depth))) return VDO_ERR_ARG;
  if (f->w < SAMP_DIV || f->h < SAMP_DIV) return VDO_ERR_ARG;         // an empty grid step: the reference's loop never ends
  if (!f->samp_pow) {
    std::vector<unsigned long long> tab(SAMP_DRAWS);
    unsigned long long s = 1ull << 32;                                  // r^-1 mod m; one MWC step multiplies by r
    for (int k = 0; k < SAMP_DRAWS; ++k) { tab[k] = s; s = (s & 0xffffffffull) * RNG_A + (s >> 32); }
    FRK(cudaMalloc(&f->samp_pow, sizeof(unsigned long long) * SAMP_DRAWS));
    FRK(cudaMemcpyAsync(f->samp_pow, tab.data(), sizeof(unsigned long long) * SAMP_DRAWS, cudaMemcpyHostToDevice, f->st));
    FRK(cudaStreamSynchronize(f->st));
  }
  const int N = VDO_SAMPLE_KEYPOINTS;
  if (int rc = ensure_scratch(f, sizeof(float) * 2 * N + sizeof(SampOut) * N + 64)) return rc;
  float* d_raw = (float*)f->scratch; SampOut* d_out = (SampOut*)(d_raw + 2 * N);
  k_sample_static<<<1, 1024, 0, f->st>>>(f->samp_pow, seed ? seed : 0xffffffffu, f->mask, f->depth, f->flow, f->w, f->h, th_depth, raw_xy ? d_raw : nullptr, d_out,
                                         f->d_count); f->launches++;
  int m = 0;
  FRK(cudaMemcpyAsync(&m, f->d_count, sizeof(int), cudaMemcpyDeviceToHost, f->st));
  if (raw_xy) FRK(cudaMemcpyAsync(raw_xy, d_raw, sizeof(float) * 2 * N, cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  m = std::min(m, max_out);
  std::vector<SampOut> h(m);
  if (m) { FRK(cudaMemcpyAsync(h.data(), d_out, sizeof(SampOut) * m, cudaMemcpyDeviceToHost, f->st)); FRK(cudaStreamSynchronize(f->st)); }
  for (int i = 0; i < m; ++i) { kx[i] = h[i].kx; ky[i] = h[i].ky; cx[i] = h[i].cx; cy[i] = h[i].cy; fu[i] = h[i].fu; fv[i] = h[i].fv; depth[i] = h[i].depth; }
  *n_out = m;
  return VDO_OK;
}

extern "C" int vdo_scene_flow(vdo_ctx* ctx, int n, const float* u_prev, const float* v_prev, const float* z_prev, const float* Tcw_prev,
                              const float* u_cur, const float* v_cur, const float* z_cur, const float* Tcw_cur, const float* K,
                              const int* label_prev, const int* label_cur, float* flow3d, float* Xw_prev, unsigned char* valid) {
  if (!ctx || n < 0) return VDO_ERR_ARG;
  if (n == 0) return VDO_OK;
  cudaStream_t st = (cudaStream_t)(uintptr_t)vdo_ctx_stream(ctx);
  const size_t fl = (size_t)n;
  static std::mutex mu; static std::map<cudaStream_t, std::pair<float*, size_t>> pool;      // grow-only scratch per stream (the call is synchronous)
  std::lock_guard<std::mutex> lk(mu);
  auto& slot = pool[st];
  const size_t need = fl * 4 * (6 + 2 + 3 + 3) + fl;
  if (need > slot.second) { cudaFree(slot.first); slot.first = nullptr; FRK(cudaMalloc(&slot.first, need * 2)); slot.second = need * 2; }
  float* d = slot.first;
  float *up = d, *vp = up + fl, *zp = vp + fl, *uc = zp + fl, *vc = uc + fl, *zc = vc + fl;
  int *lp = (int*)(zc + fl), *lc = lp + fl;
  float *df = (float*)(lc + fl), *dx = df + 3 * fl;
  unsigned char* dv = (unsigned char*)(dx + 3 * fl);
  const float* hs[6] = {u_prev, v_prev, z_prev, u_cur, v_cur, z_cur};
  for (int k = 0; k < 6; ++k) FRK(cudaMemcpyAsync(d + k * fl, hs[k], fl * 4, cudaMemcpyHostToDevice, st));
  FRK(cudaMemcpyAsync(lp, label_prev, fl * 4, cudaMemcpyHostToDevice, st));
  FRK(cudaMemcpyAsync(lc, label_cur, fl * 4, cudaMemcpyHostToDevice, st));
  Pose32 Tp, Tc;
  for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) { Tp.R[3 * r + c] = Tcw_prev[4 * r + c]; Tc.R[3 * r + c] = Tcw_cur[4 * r + c]; } Tp.t[r] = Tcw_prev[4 * r + 3]; Tc.t[r] = Tcw_cur[4 * r + 3]; }
  k_scene_flow<<<(n + 255) / 256, 256, 0, st>>>(n, up, vp, zp, Tp, uc, vc, zc, Tc, lp, lc, make_float4(K[0], K[1], K[2], K[3]), df, dx, dv);
  FRK(cudaMemcpyAsync(flow3d, df, fl * 12, cudaMemcpyDeviceToHost, st));
  if (Xw_prev) FRK(cudaMemcpyAsync(Xw_prev, dx, fl * 12, cudaMemcpyDeviceToHost, st));
  if (valid) FRK(cudaMemcpyAsync(valid, dv, fl, cudaMemcpyDeviceToHost, st));
  FRK(cudaStreamSynchronize(st));
  return VDO_OK;
}

// test hook: download pyramid level `level` (and its FAST score map) computed by the last vdo_orb_extract; sizes via w_out/h_out
extern "C" int vdo_frame_debug_level(vdo_frame* f, int level, unsigned char* img_out, unsigned char* score_out, int* w_out, int* h_out) {
  if (!f || !f->orb_ready || level < 0 || level >= f->orb.nlevels) return VDO_ERR_ARG;
  if (w_out) *w_out = f->lw[level];
  if (h_out) *h_out = f->lh[level];
  const size_t n = (size_t)f->lw[level] * f->lh[level];
  if (img_out) FRK(cudaMemcpyAsync(img_out, f->pyr[level], n, cudaMemcpyDeviceToHost, f->st));
  if (score_out) FRK(cudaMemcpyAsync(score_out, f->score[level], n, cudaMemcpyDeviceToHost, f->st));
  FRK(cudaStreamSynchronize(f->st));
  return VDO_OK;
}

// device-resident timing of the ORB front end (pyramid + score + cells) for bench/profiles: returns avg ms over reps
extern "C" int vdo_orb_time(vdo_frame* f, int reps, float* ms_avg) {
  if (!f || !f->orb_ready || reps <= 0 || !ms_avg) return VDO_ERR_ARG;
  cudaEvent_t e0, e1; FRK(cudaEventCreate(&e0)); FRK(cudaEventCreate(&e1));
  const OrbSetup& P = f->orb;
  auto run = [&]() {
    int cb = 0;
    for (int l = 0; l < P.nlevels; ++l) {
      dim3 b(32, 8), g((f->lw[l] + 31) / 32, (f->lh[l] + 7) / 8);
      if (l > 0) k_resize_u8<<<g, b, 0, f->st>>>(f->pyr[l - 1], f->lw[l - 1], f->lh[l - 1], f->pyr[l], f->lw[l], f->lh[l]);
      k_fast_score<<<g, b, 0, f->st>>>(f->pyr[l], f->lw[l], f->lh[l], f->score[l]);
    }
    (void)cb;
  };
  run();
  FRK(cudaEventRecord(e0, f->st));
  for (int i = 0; i < reps; ++i) run();
  FRK(cudaEventRecord(e1, f->st));
  FRK(cudaEventSynchronize(e1));
  float ms = 0; FRK(cudaEventElapsedTime(&ms, e0, e1));
  *ms_avg = ms / reps;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return VDO_OK;
}
