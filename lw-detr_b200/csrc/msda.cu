// Multi-scale deformable attention core, forward (reference: models/ops/src/cuda/
// ms_deform_im2col_cuda.cuh:33-84 bilinear, :237-299 kernel, launcher :923-954; host glue
// ms_deform_attn_cuda.cu:20-80; module math ops/modules/ms_deform_attn.py:118-131).
//
// Two kernels, both HBM-bound byte movers without tensor cores:
//
// 1. msda_fwd_kernel - the model path.  The reference gathers 32-byte head slices from a token-major value tensor:
//    every bilinear corner is a random DRAM sector.  Here value_proj writes the value tensor HEAD-MAJOR
//    ([image][head][token][16], gemm_tc "head-major" epilogue), so everything one (image, head) can ever sample is
//    ONE contiguous slab (51 KB at 40x40).  Persistent CTAs (one per SM, 20 warps) walk the (image, head) items: the
//    slab is streamed - in bands of <= 1680 tokens - into a four-stage shared-memory ring with 1-D bulk copies
//    (cp.async.bulk + mbarrier complete_tx; measured 7.0 TB/s at this chunk size with tools/ubench/stream_rate.cu),
//    the threads (two per (query, head): half of the samples each, all 16 channels) take the bilinear corners out of
//    shared memory.  DRAM sees the value tensor exactly once, as a linear stream; the softmax over
//    the L*P logits, the sampling-location arithmetic (incl. valid ratios of padded batches) and the weighted sum
//    stay in registers; the raw projections of the NEXT item are prefetched while the current one is sampled.
//    A P3 level (80x80 = 205 KB per head) does not fit a stage: it is cut into bands of 21 rows (one halo row), each
//    sample is handled by the band that holds both of its rows.
//
// 2. msda_op_kernel - the reference operator's own interface (token-major value [B,S,M,D], explicit sampling
//    locations and attention weights, fp32 / fp16 / bf16, any D % 8 == 0): a direct gather, one thread = 8 (16-bit)
//    or 4 (fp32) channels of one (query, head), 16-byte read-only loads, all L*P*4 corner loads issued before use.
#include "msda.h"
#include "launch.h"
#include "ptx.cuh"

#include <algorithm>

namespace lwb {

static constexpr int MS_STAGES = 4;                                // slabs / bands in flight per CTA
static constexpr int MS_STAGE_TOKENS = 1680;                       // 21 rows of 80 / 42 rows of 40
static constexpr int MS_STAGE_BYTES = MS_STAGE_TOKENS * MSDA_D * 2;
static constexpr int MS_TPQ = 2;                                   // threads per (query, head): each takes half of the L*P samples
static constexpr int MS_WARPS = 20;
static constexpr int MS_THREADS = MS_WARPS * 32;                   // 640 threads = 320 queries per pass
static constexpr int MS_QPASS = MS_THREADS / MS_TPQ;
static constexpr int MS_SMEM = MS_STAGES * MS_STAGE_BYTES + 128;

__device__ __forceinline__ U4 lds16(uint32_t addr) {
  U4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
// one 32-bit word = two 16-bit values -> packed fp32 pair (low element first), on the ALU pipe (the FMA pipe is the busy one)
template <typename T> __device__ __forceinline__ uint64_t widen2(uint32_t w);
template <> __device__ __forceinline__ uint64_t widen2<__nv_bfloat16>(uint32_t w) {
  uint64_t r;
  asm("{\n\t.reg .b32 lo, hi;\n\tshl.b32 lo, %1, 16;\n\tand.b32 hi, %1, 0xffff0000;\n\tmov.b64 %0, {lo, hi};\n\t}" : "=l"(r) : "r"(w));
  return r;
}
template <> __device__ __forceinline__ uint64_t widen2<__half>(uint32_t w) {
  uint64_t r;
  asm("{\n\t.reg .b16 l, h;\n\t.reg .f32 fl, fh;\n\tmov.b32 {l, h}, %1;\n\tcvt.f32.f16 fl, l;\n\tcvt.f32.f16 fh, h;\n\tmov.b64 %0, {fl, fh};\n\t}"
      : "=l"(r) : "r"(w));
  return r;
}
__device__ __forceinline__ uint64_t shfl_xor1_b64(uint64_t v) {
  uint32_t lo = static_cast<uint32_t>(v), hi = static_cast<uint32_t>(v >> 32);
  lo = __shfl_xor_sync(0xffffffffu, lo, 1);
  hi = __shfl_xor_sync(0xffffffffu, hi, 1);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

// ncu of the earlier versions of this kernel (history in DESIGN.md 3.2; current capture: profiles/r02_ncu_msda_medium.txt) showed it bound by
// its own instruction stream and by a tail, not by memory: 735 instructions per (query, head) - a fifth of them integer
// divisions of the item / pass bookkeeping, another third register shuffling around the 16-bit -> fp32 unpack - at 36 % issue
// utilisation, with half-CTAs that each walked whole (image, head) items (3.46 items per half at medium / B = 64: 14 % tail).
// Hence:
//   * the whole CTA (20 warps) works on ONE (image, head) slab at a time; slabs stream through a 4-stage ring filled by one
//     elected thread (cp.async.bulk + mbarrier complete_tx), so up to three slabs are in flight behind the one being sampled;
//   * TWO threads per (query, head): each takes half of the L*P samples (all 16 channels), the pair exchanges halves of its
//     partial sums with 8 shuffles and each stores 8 channels - 600 of 640 threads busy at nq = 300;
//   * item / image / head counters are incremental (no division in any loop), the unpack is two ALU operations per pair,
//     the accumulation runs on packed fp32x2 FMAs.
template <typename T, int NL, int NP>   // levels, points per head and level
__global__ void __launch_bounds__(MS_THREADS, 1) msda_fwd_kernel(const __grid_constant__ MsdaArgs p) {
  constexpr int LP = NL * NP;
  constexpr int SPT = LP / MS_TPQ;                             // samples per thread: i = sub + 2*k (levels stay balanced)
  static_assert(LP % MS_TPQ == 0 && NP % MS_TPQ == 0, "samples split evenly between the two threads of a query");
  extern __shared__ __align__(128) uint8_t ms_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(ms_smem + MS_STAGES * MS_STAGE_BYTES);
  uint64_t* empty = full + MS_STAGES;
  const int lane = threadIdx.x & 31;
  const int sub = threadIdx.x & 1;                              // which half of the samples / which 8 channels are stored
  const int qt = threadIdx.x >> 1;                              // query index inside a pass
  if (threadIdx.x == 0) {
    for (int s = 0; s < MS_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], MS_WARPS);
    }
    fence_mbar_init();
  }
  __syncthreads();
  pdl_sync();   // programmatic dependent launch: release the successor, wait for the predecessor (launch.h)
  const int nitems = p.batch * p.heads;
  const int npass = (p.nq + MS_QPASS - 1) / MS_QPASS;
  const int first = static_cast<int>(blockIdx.x), stride = static_cast<int>(gridDim.x);
  const int n_my = first < nitems ? (nitems - first + stride - 1) / stride : 0;
  const int db = stride / p.heads, dm = stride - db * p.heads;  // item += stride  <=>  (b, m) += (db, dm) with carry
  const int total = n_my * npass * p.nbands;                    // (item, pass, band) steps of this CTA
  const uint32_t smem0 = smem_u32(ms_smem);

  // ---- producer state (thread 0): next step to load
  int ld_t = 0, ld_k = 0, ld_pass = 0, ld_b = first / p.heads, ld_m = first - (first / p.heads) * p.heads;
  uint32_t ld_st = 0, ld_ph = 0;
  auto issue_load = [&]() {                                    // step ld_t -> stage ld_st
    if (ld_t >= MS_STAGES) mbar_wait(&empty[ld_st], ld_ph ^ 1u);
    const T* slab = reinterpret_cast<const T*>(p.value) + static_cast<long long>(ld_b) * p.v_b_stride + static_cast<long long>(ld_m) * p.S * MSDA_D;
    const uint32_t bytes = static_cast<uint32_t>(p.bands[ld_k].bytes);
    mbar_arrive_expect_tx(&full[ld_st], bytes);
    bulk_load(ms_smem + ld_st * MS_STAGE_BYTES, slab + static_cast<long long>(p.bands[ld_k].tok0) * MSDA_D, bytes, &full[ld_st]);
    ++ld_t;
    if (++ld_st == MS_STAGES) {
      ld_st = 0;
      ld_ph ^= 1u;
    }
    if (++ld_k == p.nbands) {
      ld_k = 0;
      if (++ld_pass == npass) {
        ld_pass = 0;
        ld_m += dm;
        ld_b += db;
        if (ld_m >= p.heads) {
          ld_m -= p.heads;
          ++ld_b;
        }
      }
    }
  };
  const bool producer = threadIdx.x == 0;
  if (producer) {
    for (int i = 0; i < MS_STAGES - 1 && ld_t < total; ++i) issue_load();
  }

  struct Raw {
    uint32_t off[SPT];         // (dx, dy) 16-bit pairs of this thread's samples
    uint32_t lg[LP / 2];       // all logits of the (query, head), 16-bit pairs
    float4 ref;
  };
  auto load_raw = [&](int b, int m, int q, Raw& r) {
    if (q >= p.nq) return;
    const long long row = static_cast<long long>(b) * p.nq + q;
    const T* oa = reinterpret_cast<const T*>(p.offs_logits) + row * p.ld_ol;
    const uint32_t* o32 = reinterpret_cast<const uint32_t*>(oa + m * (2 * LP));
#pragma unroll
    for (int k = 0; k < SPT; ++k) r.off[k] = __ldg(o32 + sub + MS_TPQ * k);
    const uint32_t* l32 = reinterpret_cast<const uint32_t*>(oa + p.heads * (2 * LP) + m * LP);
#pragma unroll
    for (int i = 0; i < LP / 2; ++i) r.lg[i] = __ldg(l32 + i);
    r.ref = __ldg(reinterpret_cast<const float4*>(p.ref) + row);
  };

  int b = first / p.heads, m = first - b * p.heads;
  // the raw projections of the NEXT (item, pass) are prefetched while the current one is sampled
  Raw nxt;
  if (n_my > 0) load_raw(b, m, qt, nxt);
  uint32_t c_st = 0, c_ph = 0;                                  // consumer stage / phase
  int t = 0;
  for (int it = 0; it < n_my; ++it) {
    int nb = b + db, nm = m + dm;
    if (nm >= p.heads) {
      nm -= p.heads;
      ++nb;
    }
    for (int pass = 0; pass < npass; ++pass) {
      const int q = pass * MS_QPASS + qt;
      const bool active = q < p.nq;
      Raw cur = nxt;
      if (pass + 1 < npass) load_raw(b, m, q + MS_QPASS, nxt);
      else if (it + 1 < n_my) load_raw(nb, nm, qt, nxt);
      // ---- this thread's samples, prepared ONCE per (item, pass) - not per band: the four corner weights (softmax weight and
      // the zero weight of out-of-image corners folded in), the clamped corner tokens relative to the level, the sample's row
      float wc[SPT][4];
      uint32_t info[SPT];     // bits 0-13: token of the (clamped) top-left corner in its level, 14: x step, 15: y step, 16-31: floor(y) + 1 (0xffff: no weight)
      if (active) {
        float lg[LP];
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < LP / 2; ++i) {
          const float2 f = Cvt<T>::unpack(cur.lg[i]);
          lg[2 * i] = f.x;
          lg[2 * i + 1] = f.y;
          mx = fmaxf(mx, fmaxf(f.x, f.y));
        }
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < LP; ++i) {
          lg[i] = __expf(lg[i] - mx);
          sum += lg[i];
        }
        const float inv = __fdividef(1.f, sum);
        const float sx = cur.ref.z * (0.5f / NP), sy = cur.ref.w * (0.5f / NP);
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
          const int l = k / (NP / MS_TPQ);                                 // sample i = sub + 2k lies in level i / NP = k / (NP / 2)
          const float2 o = Cvt<T>::unpack(cur.off[k]);
          float lx = cur.ref.x + o.x * sx, ly = cur.ref.y + o.y * sy;      // ms_deform_attn.py:125-127
          if (p.valid_ratio != nullptr) {                                  // transformer.py:352-353: boxes scaled per level
            lx *= __ldg(p.valid_ratio + (b * NL + l) * 2);
            ly *= __ldg(p.valid_ratio + (b * NL + l) * 2 + 1);
          }
          const int H = p.lvl_h[l], W = p.lvl_w[l];
          const float px = lx * W - 0.5f, py = ly * H - 0.5f;              // cuh:285-286
          const bool in = py > -1.f && px > -1.f && py < H && px < W;      // cuh:288
          const float w = in ? (sub ? lg[2 * k + 1] : lg[2 * k]) * inv : 0.f;
          const float yf = floorf(py), xf = floorf(px);
          const int y0 = static_cast<int>(yf), x0 = static_cast<int>(xf);
          const float fy = py - yf, fx = px - xf;
          // clamped corner tokens (always readable), zero weight for the corners outside the image (cuh:58-84)
          const int ya = max(y0, 0), yb = min(y0 + 1, H - 1), xa = max(x0, 0), xb = min(x0 + 1, W - 1);
          const float wy0 = y0 >= 0 ? w - w * fy : 0.f, wy1 = y0 + 1 < H ? w * fy : 0.f;
          const float wx0 = x0 >= 0 ? 1.f - fx : 0.f, wx1 = x0 + 1 < W ? fx : 0.f;
          wc[k][0] = wy0 * wx0; wc[k][1] = wy0 * wx1; wc[k][2] = wy1 * wx0; wc[k][3] = wy1 * wx1;
          info[k] = static_cast<uint32_t>(ya * W + xa) | (static_cast<uint32_t>(xb - xa) << 14) | (static_cast<uint32_t>(yb - ya) << 15) |
                    ((w != 0.f ? static_cast<uint32_t>(y0 + 1) : 0xffffu) << 16);   // a sample without weight never matches a band
        }
      }
      uint64_t acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = f2_pack(0.f, 0.f);
      for (int k = 0; k < p.nbands; ++k, ++t) {
        const int own0 = p.bands[k].own0, own1 = p.bands[k].own1, row0 = p.bands[k].row0, blvl = p.bands[k].level;
        if (producer && t + MS_STAGES - 1 < total) issue_load();           // keep three loads in flight behind this one
        mbar_wait(&full[c_st], c_ph);
        if (active) {
          const uint32_t stage = smem0 + c_st * MS_STAGE_BYTES;
#pragma unroll
          for (int ks = 0; ks < SPT; ++ks) {
            const int l = ks / (NP / MS_TPQ);
            if (NL > 1 && l != blvl) continue;                             // uniform
            const int y0 = static_cast<int>(info[ks] >> 16) - 1;
            if (y0 < own0 || y0 > own1) continue;                          // the band that holds both rows of the sample takes it
            const int W = p.lvl_w[l];
            const uint32_t a00 = stage + static_cast<uint32_t>(static_cast<int>(info[ks] & 0x3fffu) - row0 * W) * 32u;
            const uint32_t ax = ((info[ks] >> 14) & 1u) * 32u, ay = ((info[ks] >> 15) & 1u) * static_cast<uint32_t>(W) * 32u;
            const uint32_t addr[4] = {a00, a00 + ax, a00 + ay, a00 + ay + ax};
#pragma unroll
            for (int rowp = 0; rowp < 2; ++rowp) {                         // the two corners of one image row at a time (16 registers in flight)
              const U4 v[4] = {lds16(addr[rowp * 2]), lds16(addr[rowp * 2] + 16), lds16(addr[rowp * 2 + 1]), lds16(addr[rowp * 2 + 1] + 16)};
#pragma unroll
              for (int cx = 0; cx < 2; ++cx) {
                const uint64_t w2 = f2_pack(wc[ks][rowp * 2 + cx], wc[ks][rowp * 2 + cx]);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                  const U4 u = v[cx * 2 + hh];
                  const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                  for (int j = 0; j < 4; ++j) acc[hh * 4 + j] = f2_fma(w2, widen2<T>(uu[j]), acc[hh * 4 + j]);
                }
              }
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[c_st]);
        if (++c_st == MS_STAGES) {
          c_st = 0;
          c_ph ^= 1u;
        }
      }
      // ---- the pair exchanges halves: sub 0 ends up with channels 0-7, sub 1 with channels 8-15 (all lanes take part)
      uint64_t mine[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint64_t give = sub ? acc[j] : acc[4 + j];                   // what the partner stores
        const uint64_t got = shfl_xor1_b64(give);
        mine[j] = f2_add(sub ? acc[4 + j] : acc[j], got);
      }
      if (active) {
        U4 o;
        float a0, a1;
        f2_unpack(mine[0], a0, a1); o.x = Cvt<T>::pack(a0, a1);
        f2_unpack(mine[1], a0, a1); o.y = Cvt<T>::pack(a0, a1);
        f2_unpack(mine[2], a0, a1); o.z = Cvt<T>::pack(a0, a1);
        f2_unpack(mine[3], a0, a1); o.w = Cvt<T>::pack(a0, a1);
        const long long row = static_cast<long long>(b) * p.nq + q;
        *reinterpret_cast<U4*>(reinterpret_cast<T*>(p.out) + row * p.ld_out + m * MSDA_D + sub * 8) = o;
      }
    }
    b = nb;
    m = nm;
  }
}

int msda_plan(MsdaArgs* a) {
  a->nbands = 0;
  for (int l = 0; l < a->levels; ++l) {
    const int H = a->lvl_h[l], W = a->lvl_w[l];
    if (H < 1 || W < 1 || 2 * W > MS_STAGE_TOKENS || H * W > 16384 || H > 0xfff0) return -2;   // 14-bit token / 16-bit row fields of the packed sample info
    const int rows_max = MS_STAGE_TOKENS / W;                    // rows a stage holds
    if (H <= rows_max) {
      if (a->nbands >= MSDA_MAX_BANDS) return -2;
      a->bands[a->nbands++] = MsdaBand{l, 0, -1, H - 1, a->lvl_start[l], H * W * MSDA_D * 2};
      continue;
    }
    const int own = rows_max - 1;                                // one halo row per band
    for (int r0 = 0; r0 < H; r0 += own) {
      if (a->nbands >= MSDA_MAX_BANDS) return -2;
      const int r1 = std::min(r0 + own, H - 1);                  // last staged row (halo included)
      const bool last = r0 + own >= H;
      a->bands[a->nbands++] = MsdaBand{l, r0, r0 == 0 ? -1 : r0, last ? H - 1 : r0 + own - 1, a->lvl_start[l] + r0 * W, (r1 - r0 + 1) * W * MSDA_D * 2};
    }
  }
  return 0;
}

template <typename T, int NL, int NP>
static int launch_fwd(const MsdaArgs& a, cudaStream_t st) {
  int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(msda_fwd_kernel<T, NL, NP>), MS_SMEM);
  if (e) return e;
  const int items = a.batch * a.heads;
  const unsigned grid = static_cast<unsigned>(std::min(items, current_device_sms()));
  launch_k(msda_fwd_kernel<T, NL, NP>, dim3(grid), dim3(MS_THREADS), static_cast<size_t>(MS_SMEM), st, a);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
static int dispatch(const MsdaArgs& a, cudaStream_t st) {
  if (a.levels == 1 && a.points == 2) return launch_fwd<T, 1, 2>(a, st);
  if (a.levels == 2 && a.points == 4) return launch_fwd<T, 2, 4>(a, st);
  if (a.levels == 1 && a.points == 4) return launch_fwd<T, 1, 4>(a, st);
  if (a.levels == 2 && a.points == 2) return launch_fwd<T, 2, 2>(a, st);
  if (a.levels == 4 && a.points == 4) return launch_fwd<T, 4, 4>(a, st);
  return -2;
}

int msda_launch(int dtype, const MsdaArgs& a, cudaStream_t st) {
  if (a.nbands < 1 || a.batch < 1 || a.nq < 1) return -2;
  return dtype == DT_BF16 ? dispatch<__nv_bfloat16>(a, st) : dispatch<__half>(a, st);
}

// ------------------------------------------------------------------------------------------------------------------
// Operator boundary: ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
// (ms_deform_attn.h:19-35 -> ms_deform_attn_cuda.cu:20-80 -> cuh:237-299).  Same arithmetic and the same operation
// order as the reference's bilinear (cuh:33-84): val = w1 v1 + w2 v2 + w3 v3 + w4 v4; col += val * attn_weight.
template <typename T> struct Elt;
template <> struct Elt<float> {
  static constexpr int VEC = 4;
  static __device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void unpack(const U4& u, float (&f)[4]) {
    f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w);
  }
  static __device__ __forceinline__ void store(float* p, const float (&f)[4]) { *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]); }
};
template <> struct Elt<__half> {
  static constexpr int VEC = 8;
  static __device__ __forceinline__ float ld(const __half* p) { return __half2float(__ldg(p)); }
  static __device__ __forceinline__ void unpack(const U4& u, float (&f)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 t = Cvt<__half>::unpack(w[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
  }
  static __device__ __forceinline__ void store(__half* p, const float (&f)[8]) {
    U4 o; o.x = Cvt<__half>::pack(f[0], f[1]); o.y = Cvt<__half>::pack(f[2], f[3]); o.z = Cvt<__half>::pack(f[4], f[5]); o.w = Cvt<__half>::pack(f[6], f[7]);
    *reinterpret_cast<U4*>(p) = o;
  }
};
template <> struct Elt<__nv_bfloat16> {
  static constexpr int VEC = 8;
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
  static __device__ __forceinline__ void unpack(const U4& u, float (&f)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 t = Cvt<__nv_bfloat16>::unpack(w[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    U4 o; o.x = Cvt<__nv_bfloat16>::pack(f[0], f[1]); o.y = Cvt<__nv_bfloat16>::pack(f[2], f[3]); o.z = Cvt<__nv_bfloat16>::pack(f[4], f[5]); o.w = Cvt<__nv_bfloat16>::pack(f[6], f[7]);
    *reinterpret_cast<U4*>(p) = o;
  }
};

__device__ __forceinline__ U4 ldg_nc16(const void* p) {
  U4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

template <typename T>
__global__ void __launch_bounds__(256) msda_op_kernel(const MsdaOpArgs p) {
  pdl_sync();
  constexpr int VEC = Elt<T>::VEC;
  const int groups = p.D / VEC;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int g = static_cast<int>(gid % groups);
  const long long qm = gid / groups;                      // (b*Lq + q)*M + m
  if (qm >= static_cast<long long>(p.B) * p.Lq * p.M) return;
  const int m = static_cast<int>(qm % p.M);
  const long long bq = qm / p.M;
  const int b = static_cast<int>(bq / p.Lq);
  const int LP = p.L * p.P;
  const T* loc = reinterpret_cast<const T*>(p.sampling_loc) + qm * LP * 2;
  const T* aw = reinterpret_cast<const T*>(p.attn_weight) + qm * LP;
  const long long row_stride = static_cast<long long>(p.M) * p.D;            // elements between tokens
  const T* vb = reinterpret_cast<const T*>(p.value) + static_cast<long long>(b) * p.S * row_stride + m * p.D + g * VEC;
  float col[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) col[j] = 0.f;
  for (int l = 0; l < p.L; ++l) {
    const int H = static_cast<int>(__ldg(p.spatial_shapes + 2 * l)), W = static_cast<int>(__ldg(p.spatial_shapes + 2 * l + 1));
    const T* vl = vb + __ldg(p.level_start_index + l) * row_stride;
    for (int pt = 0; pt < p.P; ++pt) {
      const int i = l * p.P + pt;
      const float w_im = Elt<T>::ld(loc + 2 * i) * W - 0.5f, h_im = Elt<T>::ld(loc + 2 * i + 1) * H - 0.5f;   // cuh:285-286
      const float weight = Elt<T>::ld(aw + i);
      if (!(h_im > -1.f && w_im > -1.f && h_im < H && w_im < W)) continue;                                     // cuh:288
      const float hf = floorf(h_im), wf = floorf(w_im);
      const int h_low = static_cast<int>(hf), w_low = static_cast<int>(wf), h_high = h_low + 1, w_high = w_low + 1;
      const float lh = h_im - hf, lw = w_im - wf, hh = 1.f - lh, hw = 1.f - lw;
      const bool t = h_low >= 0, bt = h_high <= H - 1, lf = w_low >= 0, rt = w_high <= W - 1;
      const U4 zero{0u, 0u, 0u, 0u};
      // issue every corner load first (clamped addresses are always in range), then combine as cuh:58-84
      const int hc0 = max(h_low, 0), hc1 = min(h_high, H - 1), wc0 = max(w_low, 0), wc1 = min(w_high, W - 1);
      const U4 r1 = ldg_nc16(vl + (static_cast<long long>(hc0) * W + wc0) * row_stride);
      const U4 r2 = ldg_nc16(vl + (static_cast<long long>(hc0) * W + wc1) * row_stride);
      const U4 r3 = ldg_nc16(vl + (static_cast<long long>(hc1) * W + wc0) * row_stride);
      const U4 r4 = ldg_nc16(vl + (static_cast<long long>(hc1) * W + wc1) * row_stride);
      float v1[VEC], v2[VEC], v3[VEC], v4[VEC];
      Elt<T>::unpack((t && lf) ? r1 : zero, v1);
      Elt<T>::unpack((t && rt) ? r2 : zero, v2);
      Elt<T>::unpack((bt && lf) ? r3 : zero, v3);
      Elt<T>::unpack((bt && rt) ? r4 : zero, v4);
      const float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
#pragma unroll
      for (int j = 0; j < VEC; ++j) col[j] += (w1 * v1[j] + w2 * v2[j] + w3 * v3[j] + w4 * v4[j]) * weight;
    }
  }
  Elt<T>::store(reinterpret_cast<T*>(p.out) + qm * p.D + g * VEC, col);
}

// Any head dim (models/ops/test.py runs D = 2 and odd channel counts): one thread per output channel, scalar loads.
template <typename T>
__global__ void __launch_bounds__(256) msda_op_scalar_kernel(const MsdaOpArgs p) {
  pdl_sync();
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c = static_cast<int>(gid % p.D);
  const long long qm = gid / p.D;
  if (qm >= static_cast<long long>(p.B) * p.Lq * p.M) return;
  const int m = static_cast<int>(qm % p.M);
  const int b = static_cast<int>(qm / p.M / p.Lq);
  const int LP = p.L * p.P;
  const T* loc = reinterpret_cast<const T*>(p.sampling_loc) + qm * LP * 2;
  const T* aw = reinterpret_cast<const T*>(p.attn_weight) + qm * LP;
  const long long row_stride = static_cast<long long>(p.M) * p.D;
  const T* vb = reinterpret_cast<const T*>(p.value) + static_cast<long long>(b) * p.S * row_stride + m * p.D + c;
  float col = 0.f;
  for (int l = 0; l < p.L; ++l) {
    const int H = static_cast<int>(__ldg(p.spatial_shapes + 2 * l)), W = static_cast<int>(__ldg(p.spatial_shapes + 2 * l + 1));
    const T* vl = vb + __ldg(p.level_start_index + l) * row_stride;
    for (int pt = 0; pt < p.P; ++pt) {
      const int i = l * p.P + pt;
      const float w_im = Elt<T>::ld(loc + 2 * i) * W - 0.5f, h_im = Elt<T>::ld(loc + 2 * i + 1) * H - 0.5f;
      const float weight = Elt<T>::ld(aw + i);
      if (!(h_im > -1.f && w_im > -1.f && h_im < H && w_im < W)) continue;
      const float hf = floorf(h_im), wf = floorf(w_im);
      const int h_low = static_cast<int>(hf), w_low = static_cast<int>(wf), h_high = h_low + 1, w_high = w_low + 1;
      const float lh = h_im - hf, lw = w_im - wf, hh = 1.f - lh, hw = 1.f - lw;
      const float v1 = (h_low >= 0 && w_low >= 0) ? Elt<T>::ld(vl + (static_cast<long long>(h_low) * W + w_low) * row_stride) : 0.f;
      const float v2 = (h_low >= 0 && w_high <= W - 1) ? Elt<T>::ld(vl + (static_cast<long long>(h_low) * W + w_high) * row_stride) : 0.f;
      const float v3 = (h_high <= H - 1 && w_low >= 0) ? Elt<T>::ld(vl + (static_cast<long long>(h_high) * W + w_low) * row_stride) : 0.f;
      const float v4 = (h_high <= H - 1 && w_high <= W - 1) ? Elt<T>::ld(vl + (static_cast<long long>(h_high) * W + w_high) * row_stride) : 0.f;
      col += (hh * hw * v1 + hh * lw * v2 + lh * hw * v3 + lh * lw * v4) * weight;
    }
  }
  T* o = reinterpret_cast<T*>(p.out) + qm * p.D + c;
  if constexpr (sizeof(T) == 4) *o = col;
  else *o = Cvt<T>::from_f(col);
}

template <typename T>
static int launch_op(const MsdaOpArgs& a, cudaStream_t st) {
  if (a.D % Elt<T>::VEC != 0 || (reinterpret_cast<uintptr_t>(a.value) & 15) || (reinterpret_cast<uintptr_t>(a.out) & 15)) {
    const long long threads = static_cast<long long>(a.B) * a.Lq * a.M * a.D;
    launch_k(msda_op_scalar_kernel<T>, dim3(static_cast<unsigned>((threads + 255) / 256)), dim3(256), 0, st, a);
    return static_cast<int>(cudaGetLastError());
  }
  const long long threads = static_cast<long long>(a.B) * a.Lq * a.M * (a.D / Elt<T>::VEC);
  const unsigned grid = static_cast<unsigned>((threads + 255) / 256);
  launch_k(msda_op_kernel<T>, dim3(grid), dim3(256), 0, st, a);
  return static_cast<int>(cudaGetLastError());
}

// Backward of the operator (ms_deform_attn.h:37-60 -> ms_deform_attn_cuda.cu:83-154 -> cuh:301-920), fp32.
// The reference needs six kernel variants because it spends one thread per channel and must reduce the sampling-location
// and attention-weight gradients across the channels of a (query, head, level, point) through shared memory.  Here one
// thread owns a whole (query, head): it walks the D channels of every sample itself, so those two gradients are plain
// register sums (written once, no atomics, no block reduction); only grad_value, which many queries scatter into, uses
// atomicAdd - as in the reference (cuh:130-152).
__global__ void __launch_bounds__(128) msda_op_backward_kernel(const MsdaOpArgs p, const float* __restrict__ grad_out,
                                                               float* __restrict__ grad_value, float* __restrict__ grad_loc,
                                                               float* __restrict__ grad_aw) {
  const long long qm = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;        // (b*Lq + q)*M + m
  if (qm >= static_cast<long long>(p.B) * p.Lq * p.M) return;
  const int m = static_cast<int>(qm % p.M);
  const int b = static_cast<int>(qm / p.M / p.Lq);
  const int LP = p.L * p.P, D = p.D;
  const float* loc = reinterpret_cast<const float*>(p.sampling_loc) + qm * LP * 2;
  const float* aw = reinterpret_cast<const float*>(p.attn_weight) + qm * LP;
  const long long row_stride = static_cast<long long>(p.M) * D;
  const long long voff = static_cast<long long>(b) * p.S * row_stride + m * D;
  const float* vb = reinterpret_cast<const float*>(p.value) + voff;
  float* gvb = grad_value + voff;
  const float* go = grad_out + qm * D;
  for (int l = 0; l < p.L; ++l) {
    const int H = static_cast<int>(__ldg(p.spatial_shapes + 2 * l)), W = static_cast<int>(__ldg(p.spatial_shapes + 2 * l + 1));
    const long long lvl = __ldg(p.level_start_index + l) * row_stride;
    for (int pt = 0; pt < p.P; ++pt) {
      const int i = l * p.P + pt;
      const float w_im = __ldg(loc + 2 * i) * W - 0.5f, h_im = __ldg(loc + 2 * i + 1) * H - 0.5f;
      const float weight = __ldg(aw + i);
      float g_w = 0.f, g_h = 0.f, g_a = 0.f;
      if (h_im > -1.f && w_im > -1.f && h_im < H && w_im < W) {
        const float hf = floorf(h_im), wf = floorf(w_im);
        const int h_low = static_cast<int>(hf), w_low = static_cast<int>(wf), h_high = h_low + 1, w_high = w_low + 1;
        const float lh = h_im - hf, lw = w_im - wf, hh = 1.f - lh, hw = 1.f - lw;
        const bool ok1 = h_low >= 0 && w_low >= 0, ok2 = h_low >= 0 && w_high <= W - 1;
        const bool ok3 = h_high <= H - 1 && w_low >= 0, ok4 = h_high <= H - 1 && w_high <= W - 1;
        const long long o1 = lvl + (static_cast<long long>(h_low) * W + w_low) * row_stride, o2 = o1 + row_stride;
        const long long o3 = o1 + static_cast<long long>(W) * row_stride, o4 = o3 + row_stride;
        const float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
        for (int c = 0; c < D; ++c) {
          const float top = __ldg(go + c), tv = top * weight;
          const float v1 = ok1 ? __ldg(vb + o1 + c) : 0.f, v2 = ok2 ? __ldg(vb + o2 + c) : 0.f;
          const float v3 = ok3 ? __ldg(vb + o3 + c) : 0.f, v4 = ok4 ? __ldg(vb + o4 + c) : 0.f;
          // d(bilinear)/dh and /dw (cuh:112-152)
          const float dh = -hw * v1 - lw * v2 + hw * v3 + lw * v4;
          const float dw = -hh * v1 + hh * v2 - lh * v3 + lh * v4;
          g_h += dh * tv;
          g_w += dw * tv;
          g_a += top * (w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4);
          if (ok1) atomicAdd(gvb + o1 + c, w1 * tv);
          if (ok2) atomicAdd(gvb + o2 + c, w2 * tv);
          if (ok3) atomicAdd(gvb + o3 + c, w3 * tv);
          if (ok4) atomicAdd(gvb + o4 + c, w4 * tv);
        }
      }
      grad_loc[(qm * LP + i) * 2] = W * g_w;         // cuh:156-158: d/d(normalised x) = width * d/dw_im
      grad_loc[(qm * LP + i) * 2 + 1] = H * g_h;
      grad_aw[qm * LP + i] = g_a;
    }
  }
}

int msda_op_backward_launch(const MsdaOpArgs& a, const float* grad_out, float* grad_value, float* grad_loc, float* grad_aw, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(grad_value, 0, static_cast<size_t>(a.B) * a.S * a.M * a.D * sizeof(float), st);   // at::zeros_like, ms_deform_attn_cuda.cu:120
  if (e != cudaSuccess) return static_cast<int>(e);
  const long long threads = static_cast<long long>(a.B) * a.Lq * a.M;
  msda_op_backward_kernel<<<static_cast<unsigned>((threads + 127) / 128), 128, 0, st>>>(a, grad_out, grad_value, grad_loc, grad_aw);
  return static_cast<int>(cudaGetLastError());
}

int msda_op_launch(int etype, const MsdaOpArgs& a, cudaStream_t st) {
  if (etype == MSDA_ET_F32) return launch_op<float>(a, st);
  if (etype == MSDA_ET_F16) return launch_op<__half>(a, st);
  if (etype == MSDA_ET_BF16) return launch_op<__nv_bfloat16>(a, st);
  return -2;
}

}  // namespace lwb
