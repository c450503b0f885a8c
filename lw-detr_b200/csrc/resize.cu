// Pillow-exact bilinear resize of uint8 RGB frames of any size, fused with ToTensor / Normalize and the patch gather.
//
// Every caller of the reference resizes on the host before the model sees an image: demo/demo.py:146-159 runs
// torchvision's Resize([640, 640]) on a PIL image, and the eval transform with square_resize_div_64
// (datasets/transforms.py:223-232, datasets/coco.py:149-153) is the same call.  Both end in Pillow's
// Image.resize((R, R), BILINEAR).  This kernel reproduces it bit for bit (libImaging/Resample.c) on the device:
//
//   coefficients, per output index xx, in IEEE double and in this order:
//     scale = n_in / n_out;  fs = max(scale, 1);  support = fs;  ss = 1 / fs
//     c = (xx + 0.5) * scale;  xmin = max(trunc(c - support + 0.5), 0);  n = min(trunc(c + support + 0.5), n_in) - xmin
//     w[x] = max(0, 1 - |(x + xmin - c + 0.5) * ss|),  ww = w[0] + w[1] + ... (in order),  w[x] /= ww
//     k[x] = trunc(0.5 + w[x] * 2^22)   (22-bit fixed point; bilinear weights are never negative)
//   one pass:  out[i] = clamp((2^21 + sum_x src[xmin_i + x] * k_i[x]) >> 22, 0, 255)   (int32, exact)
//   order:     horizontal pass, then vertical pass on its uint8 output.  Image.resize turns the order round for very tall
//              images (height > 100 * width and a smaller target height): vertical first, then horizontal.
// An identity size needs no special case: the formula gives the taps {2^22, 0}.  Every double operation is spelled
// with an explicit rounding intrinsic so that nvcc cannot contract a product and a sum into one FMA.
//
// After the resize comes patch_gather_u8_kernel's normalisation, (u/255 - mean[c]) / std[c] in fp32 with IEEE
// divisions, so the patch matrix is bit-identical to patch_gather_u8 on the Pillow-resized frame.
//
// Shape: one CTA owns a 16 x 64 tile of output pixels (one patch row of four patches) of one image.  It computes the
// coefficients of its 64 columns and 16 rows into shared memory.  Horizontal first: it stages the source rows the tile's
// vertical taps reach, in chunks, as one RGBX word per pixel (coalesced byte loads), and runs the horizontal pass out of
// shared memory into an RGBX intermediate; vertical first (tall frames): it runs the vertical pass straight from the
// source.  The second pass writes a uint8 output tile, which is normalised and stored as 192 32-byte patch rows.
// Neighbouring tiles recompute the few intermediate values they share; those values are exact integers, so the
// recomputation cannot change a bit.  The kernel is bound by HBM: it reads each source byte about once (the overlaps hit
// L2) and writes the patch matrix once.
#include "resize.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "gemm_tc.h"
#include "launch.h"
#include "ptx.cuh"

namespace lwb {

namespace {

constexpr int TILE_H = 16, TILE_W = 64;                // output pixels per CTA: one patch row of four patches
constexpr int RS_THREADS = 256;
constexpr int OUT_PITCH = TILE_W * 3 + 4;              // bytes per output-tile row; 49 words: rows fall on different banks
constexpr int RS_SMEM_MAX = 128 * 1024;                // largest request: 8192 x 8192 -> 448 needs 120 204 bytes
constexpr int STAGE_WORDS = 6144;                      // 24 KB of staged source pixels per chunk of rows

struct ResizeParams {
  float mean[3], stdv[3];
  int R;
  int KH, KV;          // coefficient slots per output column / row (largest ksize of the batch)
  int inter_words;     // RGBX words of the first-pass buffer
  int stage_words;     // RGBX words of the source staging buffer (horizontal-first frames)
};

template <int NMAX>
struct FrameList {
  lwdetr_frame f[NMAX];
};

// Pillow's bilinear filter at (x + xmin - c + 0.5) * ss
__device__ __forceinline__ double pil_tap(int x, int xmin, double c, double ss) {
  double a = __dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(x + xmin), c), 0.5), ss);
  a = fabs(a);
  return a < 1.0 ? __dsub_rn(1.0, a) : 0.0;
}

// precompute_coeffs + normalize_coeffs_8bpc of Resample.c for one output index
__device__ void pil_coeffs(int n_in, int n_out, int xx, int kmax, int* xmin_out, int* n_taps, int* k) {
  const double scale = __ddiv_rn(static_cast<double>(n_in), static_cast<double>(n_out));
  const double fs = scale < 1.0 ? 1.0 : scale;   // filterscale; the bilinear support is 1
  const double support = fs;
  const double ss = __ddiv_rn(1.0, fs);
  const double c = __dmul_rn(__dadd_rn(static_cast<double>(xx), 0.5), scale);
  int xmin = __double2int_rz(__dadd_rn(__dsub_rn(c, support), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(c, support), 0.5));
  if (xmax > n_in) xmax = n_in;
  const int n = min(xmax - xmin, kmax);   // xmax - xmin <= 2 * ceil(support) + 1 = kmax already
  double ww = 0.0;
  for (int x = 0; x < n; ++x) ww = __dadd_rn(ww, pil_tap(x, xmin, c, ss));
  for (int x = 0; x < n; ++x) {
    double w = pil_tap(x, xmin, c, ss);
    if (ww != 0.0) w = __ddiv_rn(w, ww);
    const double f = __dmul_rn(w, 4194304.0);   // 2^22
    k[x] = __double2int_rz(w < 0.0 ? __dadd_rn(-0.5, f) : __dadd_rn(0.5, f));
  }
  *xmin_out = xmin;
  *n_taps = n;
}

__device__ __forceinline__ uint32_t clip8(int acc) {
  const int v = acc >> 22;
  return static_cast<uint32_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

template <typename T, int NMAX>
__global__ void __launch_bounds__(RS_THREADS) resize_patch_gather_u8_kernel(const FrameList<NMAX> fl, T* __restrict__ A,
                                                                            const ResizeParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int KH = p.KH, KV = p.KV;
  int* kx = reinterpret_cast<int*>(smem);   // [TILE_W][KH] column taps
  int* ky = kx + TILE_W * KH;               // [TILE_H][KV] row taps
  int* xb = ky + TILE_H * KV;               // [TILE_W] first column, [TILE_W] column tap count
  int* yb = xb + 2 * TILE_W;                // [TILE_H] first row, [TILE_H] row tap count
  uint32_t* inter = reinterpret_cast<uint32_t*>(yb + 2 * TILE_H);   // first-pass output, one RGBX word per pixel
  uint32_t* stage = inter + p.inter_words;                         // source rows staged as RGBX words (horizontal first)
  uint8_t* otile = reinterpret_cast<uint8_t*>(stage + p.stage_words);   // [TILE_H][OUT_PITCH] resized pixels

  const int b = blockIdx.y, tid = threadIdx.x;
  const lwdetr_frame fr = fl.f[b];
  const int R = p.R, G = R / 16, tiles_x = G / 4;
  const int band = blockIdx.x / tiles_x, tx = blockIdx.x - band * tiles_x;
  const int y0 = band * TILE_H, x0 = tx * TILE_W;
  // the coefficients depend on the frame's size only: computed before waiting for the predecessor grid
  if (tid < TILE_W) pil_coeffs(fr.width, R, x0 + tid, KH, &xb[tid], &xb[TILE_W + tid], kx + tid * KH);
  else if (tid < TILE_W + TILE_H) {
    const int i = tid - TILE_W;
    pil_coeffs(fr.height, R, y0 + i, KV, &yb[i], &yb[TILE_H + i], ky + i * KV);
  }
  pdl_sync();
  __syncthreads();

  const bool vfirst = fr.height > 100 * fr.width && R < fr.height;
  const uint8_t* src = fr.data;
  const long long rs = fr.row_stride;
  const int c0 = xb[0], r0 = yb[0];
  // source columns [c0, c0 + ncols) the tile's 64 output columns reach; source rows [r0, r0 + nrows) its 16 rows reach
  const int ncols = min(xb[TILE_W - 1] + xb[2 * TILE_W - 1] - c0, vfirst ? p.inter_words / TILE_H : p.stage_words);
  const int nrows = min(yb[TILE_H - 1] + yb[2 * TILE_H - 1] - r0, p.inter_words / TILE_W);
  if (!vfirst) {
    // ---- horizontal pass, chunks of `rc` source rows: stage them as RGBX words with coalesced byte loads, then
    // inter[r][j] = taps of column j over the staged row (neighbouring threads: neighbouring columns, distinct banks)
    const int rc = p.stage_words / ncols;
    for (int q0 = 0; q0 < nrows; q0 += rc) {
      const int rows = min(rc, nrows - q0);
      for (int it = tid; it < rows * ncols; it += RS_THREADS) {
        const int r = it / ncols, x = it - r * ncols;
        const uint8_t* s = src + (r0 + q0 + r) * rs + (c0 + x) * 3;
        stage[it] = static_cast<uint32_t>(__ldg(s)) | (static_cast<uint32_t>(__ldg(s + 1)) << 8) |
                    (static_cast<uint32_t>(__ldg(s + 2)) << 16);
      }
      __syncthreads();
      for (int it = tid; it < rows * TILE_W; it += RS_THREADS) {
        const int r = it / TILE_W, j = it - r * TILE_W;
        const uint32_t* s = stage + r * ncols + (xb[j] - c0);
        const int* k = kx + j * KH;
        const int n = xb[TILE_W + j];
        int a0 = 1 << 21, a1 = 1 << 21, a2 = 1 << 21;
        for (int t = 0; t < n; ++t) {
          const uint32_t w = s[t];
          const int kt = k[t];
          a0 += static_cast<int>(w & 255u) * kt;
          a1 += static_cast<int>((w >> 8) & 255u) * kt;
          a2 += static_cast<int>(w >> 16) * kt;
        }
        inter[(q0 + r) * TILE_W + j] = clip8(a0) | (clip8(a1) << 8) | (clip8(a2) << 16);
      }
      __syncthreads();
    }
  } else {
    // ---- vertical pass straight from the source (a tall, narrow frame): inter[i][x] for the tile's 16 output rows
    for (int it = tid; it < TILE_H * ncols; it += RS_THREADS) {
      const int i = it / ncols, x = it - i * ncols;
      const uint8_t* s = src + yb[i] * rs + (c0 + x) * 3;
      const int* k = ky + i * KV;
      const int n = yb[TILE_H + i];
      int a0 = 1 << 21, a1 = 1 << 21, a2 = 1 << 21;
      for (int t = 0; t < n; ++t) {
        const int kt = k[t];
        a0 += static_cast<int>(__ldg(s)) * kt;
        a1 += static_cast<int>(__ldg(s + 1)) * kt;
        a2 += static_cast<int>(__ldg(s + 2)) * kt;
        s += rs;
      }
      inter[i * ncols + x] = clip8(a0) | (clip8(a1) << 8) | (clip8(a2) << 16);
    }
    __syncthreads();
  }

  // ---- second pass -> otile (a warp walks one output row: neighbouring columns)
  for (int it = tid; it < TILE_H * TILE_W; it += RS_THREADS) {
    const int i = it / TILE_W, j = it - i * TILE_W;
    const uint32_t* s;
    int step, n;
    const int* k;
    if (!vfirst) { s = inter + (yb[i] - r0) * TILE_W + j; step = TILE_W; k = ky + i * KV; n = yb[TILE_H + i]; }
    else { s = inter + i * ncols + (xb[j] - c0); step = 1; k = kx + j * KH; n = xb[TILE_W + j]; }
    int a0 = 1 << 21, a1 = 1 << 21, a2 = 1 << 21;
    for (int t = 0; t < n; ++t) {
      const uint32_t w = *s;
      const int kt = k[t];
      a0 += static_cast<int>(w & 255u) * kt;
      a1 += static_cast<int>((w >> 8) & 255u) * kt;
      a2 += static_cast<int>(w >> 16) * kt;
      s += step;
    }
    uint8_t* o = otile + i * OUT_PITCH + j * 3;
    o[0] = static_cast<uint8_t>(clip8(a0));
    o[1] = static_cast<uint8_t>(clip8(a1));
    o[2] = static_cast<uint8_t>(clip8(a2));
  }
  __syncthreads();

  // ---- normalise and store: thread = (patch row py, patch pp, channel c) -> one 32-byte row of the patch matrix
  if (tid < TILE_H * 12) {
    const int py = tid & 15, pc = tid >> 4, pp = pc / 3, c = pc - pp * 3;
    const uint8_t* s = otile + py * OUT_PITCH + pp * 48 + c;
    float f[16];
#pragma unroll
    for (int px = 0; px < 16; ++px) {
      const float u = static_cast<float>(s[px * 3]);
      f[px] = (u / 255.f - p.mean[c]) / p.stdv[c];             // ToTensor (/255) then Normalize, as patch_gather_u8
    }
    U8 o;
#pragma unroll
    for (int q = 0; q < 8; ++q) o.v[q] = Cvt<T>::pack(f[2 * q], f[2 * q + 1]);
    const int wh = G / 4, X = tx * 4 + pp;
    const int win = (band / wh) * 4 + X / wh, t = (band % wh) * wh + X % wh;   // window-major row (vit.py:353-358)
    const long long r = static_cast<long long>(b) * G * G + win * wh * wh + t;
    stg256(A + r * 768 + c * 256 + py * 16, o);
  }
}

// rows (or columns) of the source one tile's taps can reach: 15 (63) output steps plus both supports, rounded up
int span_bound(int n_in, int R, int steps) {
  const double s = static_cast<double>(n_in) / R, sup = std::max(s, 1.0);
  return std::min(n_in, static_cast<int>(steps * s + 2.0 * sup) + 3);
}
int ksize(int n_in, int R) { return 2 * std::max(1, (n_in + R - 1) / R) + 1; }

template <typename T, int NMAX>
int launch_frames(const lwdetr_frame* frames, int B, const ResizeParams& p, size_t smem, void* A, cudaStream_t st) {
  FrameList<NMAX> fl;
  for (int i = 0; i < B; ++i) fl.f[i] = frames[i];
  auto kern = resize_patch_gather_u8_kernel<T, NMAX>;
  if (smem > 48 * 1024) {
    const int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(kern), RS_SMEM_MAX);
    if (e) return e;
  }
  const int G = p.R / 16;
  launch_k(kern, dim3(static_cast<unsigned>(G * (G / 4)), static_cast<unsigned>(B)), dim3(RS_THREADS), smem, st, fl,
           static_cast<T*>(A), p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace

int resize_patch_gather_u8_launch(int dtype, const lwdetr_frame* frames, int B, int R, const float* mean, const float* stdv,
                                  void* A, cudaStream_t st) {
  if (R <= 0 || R % 64 != 0 || B < 1 || B > LWDETR_MAX_FRAMES) return -2;
  ResizeParams p;
  for (int c = 0; c < 3; ++c) { p.mean[c] = mean[c]; p.stdv[c] = stdv[c]; }
  p.R = R; p.KH = 1; p.KV = 1; p.inter_words = 0; p.stage_words = 0;
  for (int i = 0; i < B; ++i) {
    const lwdetr_frame& f = frames[i];
    if (!f.data || f.height < 1 || f.width < 1 || f.height > LWDETR_MAX_FRAME_SIDE || f.width > LWDETR_MAX_FRAME_SIDE ||
        f.row_stride < 3LL * f.width)
      return -2;
    p.KH = std::max(p.KH, ksize(f.width, R));
    p.KV = std::max(p.KV, ksize(f.height, R));
    const int ncols = span_bound(f.width, R, TILE_W - 1), nrows = span_bound(f.height, R, TILE_H - 1);
    if (f.height > 100 * f.width && R < f.height) {
      p.inter_words = std::max(p.inter_words, TILE_H * ncols);
    } else {
      p.inter_words = std::max(p.inter_words, TILE_W * nrows);
      p.stage_words = std::max(p.stage_words, std::min(nrows, std::max(1, STAGE_WORDS / ncols)) * ncols);
    }
  }
  const size_t smem = 4 * static_cast<size_t>(TILE_W * p.KH + TILE_H * p.KV + 2 * TILE_W + 2 * TILE_H) +
                      4 * static_cast<size_t>(p.inter_words + p.stage_words) + TILE_H * OUT_PITCH;
  if (smem > RS_SMEM_MAX) return -2;
  if (dtype == DT_BF16)
    return B <= 64 ? launch_frames<__nv_bfloat16, 64>(frames, B, p, smem, A, st) : launch_frames<__nv_bfloat16, LWDETR_MAX_FRAMES>(frames, B, p, smem, A, st);
  return B <= 64 ? launch_frames<__half, 64>(frames, B, p, smem, A, st) : launch_frames<__half, LWDETR_MAX_FRAMES>(frames, B, p, smem, A, st);
}

}  // namespace lwb
