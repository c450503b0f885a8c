// Fused multi-head attention core: O = softmax(Q K^T * scale) V, never materialising the scores.
// One kernel serves the three attention shapes of LW-DETR by viewing tokens as (sequence, position):
//   * ViT window attention : 16*B sequences of 100 tokens  (vit.py:130-137 with B' = 16B)
//   * ViT global attention : B sequences of 1600 tokens    (vit.py:201-204 + 130-137)
//   * decoder self-attention: B sequences of nq queries    (attention.py:563-606)
// thanks to the window-major token layout (vit.py:353-358) both ViT cases read the same [B*1600, 3C]
// qkv matrix with no permutation.  Q/K/V are addressed as row-major matrices with a leading
// dimension and a per-head column offset, so the packed qkv GEMM output is consumed in place.
//
// Kernels in this file (register-resident flash attention: mma.sync m16n8k16 with fp32 accumulation, K/V chunks
// in a 3-stage cp.async ring, exp2 against the running maximum of the raw scores) take what the tcgen05 kernels do not:
//   attn_kernel       - sequences longer than 112 tokens (decoder self-attention)
//   attn_short_kernel - sequences of up to 112 tokens, persistent CTAs walking (window, head) items
// Packed qkv at head dims 16 and 32 goes to the slot kernel (attn_slots.cu), long packed sequences at head dim 64 to
// attn_tc.cu (attention_launch below; measured crossovers in DESIGN.md 3.1).
#include "attn.h"
#include "launch.h"
#include "ptx.cuh"

#include <algorithm>

namespace lwb {

template <typename T> struct Mma;
template <> struct Mma<__half> {
  static __device__ __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};
template <> struct Mma<__nv_bfloat16> {
  static __device__ __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool pred) {
  const int sz = pred ? 16 : 0;   // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

static constexpr int KC = 64;      // keys per shared-memory chunk
static constexpr int NSTAGE = 3;   // K/V ring: chunk ch+2 is prefetched while ch is consumed -> one barrier per chunk

// One 64-key chunk of the online-softmax attention for a warp's 16 query rows.
//   qf: Q fragments (A operand); cK / cV: the chunk's K and V rows in shared memory ([64][LDS]);
//   kbase: index of the chunk's first key; keys >= seqlen are masked.
//   NT: 8-key n-tiles of this chunk that can hold valid keys (8 = the full 64-key chunk; the second chunk of a 100-token
//       window only needs 5: no scores, exponentials or P V steps are spent on keys that cannot exist).
template <typename T, int DH, int NT = 8>
__device__ __forceinline__ void attn_chunk(const uint32_t (&qf)[DH / 16][4], const T* cK, const T* cV, int kbase, int seqlen,
                                           float scale_log2, int lane, float (&m_run)[2], float (&lsum)[4], float (&o)[DH / 8][4]) {
  constexpr int LDS = DH + 8;
  const int t4 = lane & 3;
  const uint32_t ones2 = Cvt<T>::pack(1.f, 1.f);
    // ---- S = Q K^T for 64 keys: 8 n-tiles of 8 keys
    constexpr int NTP = (NT + 1) & ~1;   // n-tiles are produced in pairs (one ldmatrix.x4 feeds two)
    float s[NTP][4];
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
    for (int nt = 0; nt < NTP; nt += 2) {
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
        // x4 = (keys nt*8.., dh lo), (keys nt*8.., dh hi), (keys (nt+1)*8.., dh lo), (keys (nt+1)*8.., dh hi)
        uint32_t kf[4];
        const int key = (nt + (lane >> 4)) * 8 + (lane & 7);
        const int c = kk * 16 + ((lane >> 3) & 1) * 8;
        ldsm_x4(kf, smem_u32(cK + key * LDS + c));
        Mma<T>::run(s[nt], qf[kk], kf[0], kf[1]);
        Mma<T>::run(s[nt + 1], qf[kk], kf[2], kf[3]);
      }
    }
    // ---- online softmax.  Instruction diet (the kernel is MUFU/issue bound at dh = 16): the max runs on the
    // raw scores, scale and max-subtraction are one FFMA feeding ex2, tail masking only touches the last
    // chunk, and the row sums come from one extra MMA against a ones fragment (below) instead of FADDs.
    if (kbase + NT * 8 > seqlen) {
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (kbase + nt * 8 + t4 * 2 + (j & 1) >= seqlen) s[nt][j] = -INFINITY;
    }
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
    }
    float alpha[2], msc[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 1));
      mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 2));
      const float m_new = fmaxf(m_run[h], mx[h]);            // running max of the RAW scores
      alpha[h] = ex2((m_run[h] - m_new) * scale_log2);
      m_run[h] = m_new;
      msc[h] = m_new * scale_log2;
    }
    uint32_t pf[NTP / 2][4];
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt) {
      if (nt >= NT) {                                          // padding half of the last 16-key step
        pf[nt >> 1][(nt & 1) * 2 + 0] = 0u;
        pf[nt >> 1][(nt & 1) * 2 + 1] = 0u;
        continue;
      }
      const float p0 = ex2(fmaf(s[nt][0], scale_log2, -msc[0]));
      const float p1 = ex2(fmaf(s[nt][1], scale_log2, -msc[0]));
      const float p2 = ex2(fmaf(s[nt][2], scale_log2, -msc[1]));
      const float p3 = ex2(fmaf(s[nt][3], scale_log2, -msc[1]));
      // C fragments of n-tiles (2j, 2j+1) form the A fragment of key-step j
      pf[nt >> 1][(nt & 1) * 2 + 0] = Cvt<T>::pack(p0, p1);
      pf[nt >> 1][(nt & 1) * 2 + 1] = Cvt<T>::pack(p2, p3);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) lsum[j] *= alpha[j >> 1];
#pragma unroll
    for (int dt = 0; dt < DH / 8; ++dt) {
      o[dt][0] *= alpha[0];
      o[dt][1] *= alpha[0];
      o[dt][2] *= alpha[1];
      o[dt][3] *= alpha[1];
    }
    // ---- O += P V
#pragma unroll
    for (int kt = 0; kt < NTP / 2; ++kt) {
      Mma<T>::run(lsum, pf[kt], ones2, ones2);               // row sums of the rounded P, fp32 accumulate
#pragma unroll
      for (int dt = 0; dt < DH / 8; dt += 2) {
        // trans x4 = (keys 0-7, dh dt), (keys 8-15, dh dt), (keys 0-7, dh dt+1), (keys 8-15, dh dt+1)
        uint32_t vf[4];
        const int key = kt * 16 + (lane & 15);
        const int c = (dt + (lane >> 4)) * 8;
        ldsm_x4_t(vf, smem_u32(cV + key * LDS + c));
        Mma<T>::run(o[dt], pf[kt], vf[0], vf[1]);
        Mma<T>::run(o[dt + 1], pf[kt], vf[2], vf[3]);
      }
    }
}

template <typename T, int DH, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) attn_kernel(const AttnArgs p) {
  pdl_sync();   // programmatic dependent launch: release the successor, wait for the predecessor (launch.h)
  constexpr int QROWS = WARPS * 16;
  constexpr int LDS = DH + 8;            // padded row (elements): 16 B pad => conflict-free ldmatrix
  constexpr int CPR = DH / 8;            // 16-byte chunks per row
  extern __shared__ __align__(16) uint8_t smem_attn[];
  T* sQ = reinterpret_cast<T*>(smem_attn);
  T* sK = sQ + QROWS * LDS;              // [NSTAGE][KC][LDS]
  T* sV = sK + NSTAGE * KC * LDS;        // [NSTAGE][KC][LDS]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qtile = blockIdx.x, head = blockIdx.y, seq = blockIdx.z;
  const int q0 = qtile * QROWS;
  const long long row_base = static_cast<long long>(seq) * p.seqlen;
  const T* gq = reinterpret_cast<const T*>(p.q) + head * DH;
  const T* gk = reinterpret_cast<const T*>(p.k) + head * DH;
  const T* gv = reinterpret_cast<const T*>(p.v) + head * DH;

  // ---- async load of the Q tile and of K/V chunk 0
  for (int i = tid; i < QROWS * CPR; i += WARPS * 32) {
    const int r = i / CPR, c = i % CPR;
    const bool ok = (q0 + r) < p.seqlen;
    const T* src = gq + (row_base + (ok ? q0 + r : 0)) * p.ldq + c * 8;
    cp_async16(smem_u32(sQ + r * LDS + c * 8), src, ok);
  }
  auto load_kv = [&](int chunk, int buf) {
    const int k0 = chunk * KC;
    for (int i = tid; i < KC * CPR; i += WARPS * 32) {
      const int r = i / CPR, c = i % CPR;
      const bool ok = (k0 + r) < p.seqlen;
      const long long row = row_base + (ok ? k0 + r : 0);
      cp_async16(smem_u32(sK + (buf * KC + r) * LDS + c * 8), gk + row * p.ldk + c * 8, ok);
      cp_async16(smem_u32(sV + (buf * KC + r) * LDS + c * 8), gv + row * p.ldv + c * 8, ok);
    }
  };
  const int nchunks = (p.seqlen + KC - 1) / KC;
  load_kv(0, 0);
  cp_async_commit();
  if (nchunks > 1) load_kv(1, 1);
  cp_async_commit();                     // (possibly empty) group keeps the wait_group arithmetic uniform

  uint32_t qf[DH / 16][4];
  float o[DH / 8][4];
#pragma unroll
  for (int i = 0; i < DH / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY};
  float lsum[4] = {0.f, 0.f, 0.f, 0.f};                      // [row g | row g | row g+8 | row g+8] sums of P
  const int g = lane >> 2, t4 = lane & 3;

  for (int ch = 0; ch < nchunks; ++ch) {
    const int buf = ch % NSTAGE;
    cp_async_wait<1>();                  // chunk ch has landed (only the newest group may still be in flight)
    __syncthreads();                     // ... for every thread; also: everyone finished chunk ch-1
    if (ch + 2 < nchunks) load_kv(ch + 2, (ch + 2) % NSTAGE);   // refills the buffer consumed at ch-1
    cp_async_commit();
    if (ch == 0) {
      // Q fragments (A operand): ldmatrix x4 = (rows 0-7,k 0-7), (rows 8-15,k 0-7), (rows 0-7,k 8-15), (rows 8-15,k 8-15)
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
        const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        const int c = kk * 16 + (lane >> 4) * 8;
        ldsm_x4(qf[kk], smem_u32(sQ + r * LDS + c));
      }
    }
    const T* cK = sK + buf * KC * LDS;
    const T* cV = sV + buf * KC * LDS;

    attn_chunk<T, DH>(qf, cK, cV, ch * KC, p.seqlen, p.scale_log2, lane, m_run, lsum, o);
  }

  // ---- finalise: divide by the row sums, stage through this warp's Q rows, 16-byte coalesced stores
  const float l_run[2] = {1.f / lsum[0], 1.f / lsum[2]};
  T* sO = sQ + warp * 16 * LDS;
#pragma unroll
  for (int dt = 0; dt < DH / 8; ++dt) {
    *reinterpret_cast<uint32_t*>(sO + g * LDS + dt * 8 + t4 * 2) = Cvt<T>::pack(o[dt][0] * l_run[0], o[dt][1] * l_run[0]);
    *reinterpret_cast<uint32_t*>(sO + (g + 8) * LDS + dt * 8 + t4 * 2) =
        Cvt<T>::pack(o[dt][2] * l_run[1], o[dt][3] * l_run[1]);
  }
  __syncwarp();
  T* go = reinterpret_cast<T*>(p.o) + head * DH;
  for (int i = lane; i < 16 * CPR; i += 32) {
    const int r = i / CPR, c = i % CPR;
    const int qrow = q0 + warp * 16 + r;
    if (qrow < p.seqlen)
      *reinterpret_cast<U4*>(go + (row_base + qrow) * p.ldo + c * 8) = *reinterpret_cast<const U4*>(sO + r * LDS + c * 8);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Short sequences (seqlen <= 112, i.e. the 10x10 ViT windows): one work item = one (sequence, head), whose
// whole Q / K / V (<= 128 rows) fits one shared-memory buffer.  A per-item CTA spends most of its life waiting
// for its only loads, so here persistent CTAs walk items  blockIdx.x, +gridDim.x, ...  (head fastest: the CTAs
// running at the same time read neighbouring 32..128-byte slices of the same token rows) and prefetch item
// i+2 into a 3-deep buffer ring while item i is computed - the HBM latency is hidden behind the math and the
// kernel runs at the larger of its HBM time and its exp (MUFU) time.
template <typename T, int DH>
__global__ void __launch_bounds__(7 * 32) attn_short_kernel(const AttnArgs p) {
  pdl_sync();   // programmatic dependent launch: release the successor, wait for the predecessor (launch.h)
  constexpr int WARPS = 7, QROWS = 112, KROWS = 128, NBUF = 3;
  constexpr int LDS = DH + 8, CPR = DH / 8;
  constexpr int BUF_ELEMS = (QROWS + 2 * KROWS) * LDS;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  T* sbase = reinterpret_cast<T*>(smem_attn);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const long long nitems = static_cast<long long>(p.nseq) * p.heads;

  auto issue_loads = [&](long long item, int buf) {
    const int head = static_cast<int>(item % p.heads);
    const long long row_base = (item / p.heads) * p.seqlen;
    T* sQ = sbase + buf * BUF_ELEMS;
    T* sK = sQ + QROWS * LDS;
    T* sV = sK + KROWS * LDS;
    const T* gq = reinterpret_cast<const T*>(p.q) + head * DH;
    const T* gk = reinterpret_cast<const T*>(p.k) + head * DH;
    const T* gv = reinterpret_cast<const T*>(p.v) + head * DH;
    for (int i = tid; i < KROWS * CPR; i += WARPS * 32) {
      const int r = i / CPR, c = i % CPR;
      const bool ok = r < p.seqlen;
      const long long row = row_base + (ok ? r : 0);
      if (r < QROWS) cp_async16(smem_u32(sQ + r * LDS + c * 8), gq + row * p.ldq + c * 8, ok);
      cp_async16(smem_u32(sK + r * LDS + c * 8), gk + row * p.ldk + c * 8, ok);
      cp_async16(smem_u32(sV + r * LDS + c * 8), gv + row * p.ldv + c * 8, ok);
    }
  };

  long long item = blockIdx.x;
  if (item < nitems) issue_loads(item, 0);
  cp_async_commit();
  if (item + gridDim.x < nitems) issue_loads(item + gridDim.x, 1);
  cp_async_commit();

  for (int it = 0; item < nitems; item += gridDim.x, ++it) {
    const int buf = it % NBUF;
    cp_async_wait<1>();                    // this item's group has landed
    __syncthreads();                       // ... for all threads; everyone is also done with item it-1
    if (item + 2LL * gridDim.x < nitems) issue_loads(item + 2LL * gridDim.x, (it + 2) % NBUF);
    cp_async_commit();

    T* sQ = sbase + buf * BUF_ELEMS;
    const T* sK = sQ + QROWS * LDS;
    const T* sV = sK + KROWS * LDS;
    uint32_t qf[DH / 16][4];
#pragma unroll
    for (int kk = 0; kk < DH / 16; ++kk) {
      const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
      const int c = kk * 16 + (lane >> 4) * 8;
      ldsm_x4(qf[kk], smem_u32(sQ + r * LDS + c));
    }
    float o[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY};
    float lsum[4] = {0.f, 0.f, 0.f, 0.f};
    attn_chunk<T, DH>(qf, sK, sV, 0, p.seqlen, p.scale_log2, lane, m_run, lsum, o);
    if (p.seqlen > KC + 40) attn_chunk<T, DH, 6>(qf, sK + KC * LDS, sV + KC * LDS, KC, p.seqlen, p.scale_log2, lane, m_run, lsum, o);   // keys 64..111 (seqlen <= 112 here)
    else if (p.seqlen > KC) attn_chunk<T, DH, 5>(qf, sK + KC * LDS, sV + KC * LDS, KC, p.seqlen, p.scale_log2, lane, m_run, lsum, o);   // keys 64..103: the 100-token windows

    const float l_run[2] = {1.f / lsum[0], 1.f / lsum[2]};
    T* sO = sQ + warp * 16 * LDS;          // this warp's own Q rows: already consumed into qf
    __syncwarp();
#pragma unroll
    for (int dt = 0; dt < DH / 8; ++dt) {
      *reinterpret_cast<uint32_t*>(sO + g * LDS + dt * 8 + t4 * 2) = Cvt<T>::pack(o[dt][0] * l_run[0], o[dt][1] * l_run[0]);
      *reinterpret_cast<uint32_t*>(sO + (g + 8) * LDS + dt * 8 + t4 * 2) = Cvt<T>::pack(o[dt][2] * l_run[1], o[dt][3] * l_run[1]);
    }
    __syncwarp();
    const int head = static_cast<int>(item % p.heads);
    const long long row_base = (item / p.heads) * p.seqlen;
    T* go = reinterpret_cast<T*>(p.o) + head * DH;
    for (int i = lane; i < 16 * CPR; i += 32) {
      const int r = i / CPR, c = i % CPR;
      const int qrow = warp * 16 + r;
      if (qrow < p.seqlen)
        *reinterpret_cast<U4*>(go + (row_base + qrow) * p.ldo + c * 8) = *reinterpret_cast<const U4*>(sO + r * LDS + c * 8);
    }
  }
}

template <typename T, int DH>
static int launch_short(const AttnArgs& a, cudaStream_t st) {
  constexpr int LDS = DH + 8;
  const size_t smem = static_cast<size_t>(3) * (112 + 256) * LDS * sizeof(T);
  if (int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(attn_short_kernel<T, DH>), 200 * 1024)) return e;
  static int ctas_per_sm = 0;   // a property of the kernel image and the sm_100a SM, identical on every device of a B200 box
  if (!ctas_per_sm) {
    int n = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, attn_short_kernel<T, DH>, 7 * 32, smem);
    if (e != cudaSuccess) return static_cast<int>(e);
    ctas_per_sm = n > 0 ? n : 1;
  }
  const int sms = current_device_sms();
  const long long items = static_cast<long long>(a.nseq) * a.heads;
  const unsigned grid = static_cast<unsigned>(std::min<long long>(items, static_cast<long long>(sms) * ctas_per_sm));
  launch_k(attn_short_kernel<T, DH>, dim3(grid), dim3(7 * 32), smem, st, a);
  return static_cast<int>(cudaGetLastError());
}

template <typename T, int DH, int WARPS>
static int launch(const AttnArgs& a, cudaStream_t st) {
  constexpr int LDS = DH + 8;
  const size_t smem = static_cast<size_t>(WARPS * 16 + 2 * NSTAGE * KC) * LDS * sizeof(T);
  if (int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(attn_kernel<T, DH, WARPS>), 96 * 1024)) return e;
  dim3 grid((a.seqlen + WARPS * 16 - 1) / (WARPS * 16), a.heads, a.nseq);
  launch_k(attn_kernel<T, DH, WARPS>, dim3(grid), dim3(WARPS * 32), smem, st, a);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
static int dispatch(const AttnArgs& a, int dh, cudaStream_t st) {
  if (a.seqlen <= 112) {
    if (dh == 16) return launch_short<T, 16>(a, st);
    if (dh == 32) return launch_short<T, 32>(a, st);
    if (dh == 64) return launch_short<T, 64>(a, st);
    return -2;
  }
  const int warps = a.seqlen >= 1024 ? 8 : 4;
#define LWB_ATTN_CASE(D, W) if (dh == D && warps == W) return launch<T, D, W>(a, st);
  LWB_ATTN_CASE(16, 8) LWB_ATTN_CASE(16, 4)
  LWB_ATTN_CASE(32, 8) LWB_ATTN_CASE(32, 4)
  LWB_ATTN_CASE(64, 8) LWB_ATTN_CASE(64, 4)
#undef LWB_ATTN_CASE
  return -2;
}

int attention_tc_launch(int dtype, const AttnArgs& a, int dh, int C, cudaStream_t st);      // attn_tc.cu
int attention_slots_launch(int dtype, const AttnArgs& a, int dh, int C, cudaStream_t st);   // attn_slots.cu

// Packed qkv at head dims 16 and 32 -> the slot kernel (attn_slots.cu; B200, isolated, global attention: medium B=64 612 us
// against 825 us of the attn_tc.cu kernel, large B=32 334 against 424).  Long packed sequences at head dim 64 -> attn_tc.cu
// (measured 18-22 % faster than the mma.sync kernel there).  Everything else -> the mma.sync kernels above.
int attention_launch(int dtype, const AttnArgs& a, int dh, cudaStream_t st) {
  const long long dk = (static_cast<const char*>(a.k) - static_cast<const char*>(a.q)) / 2;
  const long long dv = (static_cast<const char*>(a.v) - static_cast<const char*>(a.q)) / 2;
  const bool packed = dk > 0 && dv == 2 * dk && a.ldq == a.ldk && a.ldq == a.ldv && dk == static_cast<long long>(a.heads) * dh &&
                      a.ldq >= 3 * dk && (reinterpret_cast<uintptr_t>(a.q) & 15) == 0;
  if (packed && (dh == 16 || dh == 32)) return attention_slots_launch(dtype, a, dh, static_cast<int>(dk), st);
  if (packed && a.seqlen >= 512 && dh == 64) return attention_tc_launch(dtype, a, dh, static_cast<int>(dk), st);
  return dtype == DT_BF16 ? dispatch<__nv_bfloat16>(a, dh, st) : dispatch<__half>(a, dh, st);
}

}  // namespace lwb
