// tcgen05 / TMA attention for long sequences at head dim 64 (the ViT global-attention blocks, vit.py:201-204 + 130-137;
// head dims 16 and 32 take the slot kernel in attn_slots.cu).
//
// One CTA (one per SM, all 512 TMEM columns) owns TWO 128-row query tiles of one (sequence, head).  Q, K and V
// tiles are fetched by TMA straight out of the packed [rows, 3C] qkv matrix (box = 128 rows x dh columns at
// column  part*C + head*dh, hardware swizzle matching the dh*2-byte row pitch); S = Q K^T and O = P V run on the
// tensor core with accumulators in TMEM:
//
//   warp 0      : TMA producer (both Q tiles once, then rings of 128-key K and V chunks)
//   warp 1 / 18 : tcgen05.mma issuer of query tile 0 / 1 (warp 1 also owns the TMEM allocation).
//                 S_t: A = Q_t (smem, K-major), B = K chunk (smem, K-major);
//                 O_t: A = P_t (TMEM, written by the softmax warps), B = V chunk (smem, MN-major)
//   warps 2-9   : softmax of tile 0, warps 10-17: softmax of tile 1.  TWO threads per query row (64 keys each):
//                 four softmax warps per scheduler instead of two hide the per-warp issue latency.
//
// What bounds this kernel (measured, profiles/r01e_*, r01f_ubench_tmem_rate.txt): the softmax warps' own instruction
// stream and the MUFU (16 exp/clk/SM) - not TMEM bandwidth (440-940 B/clk/SM measured) and not the tensor core (every
// tcgen05.mma with N <= 64 costs 45 clk: S + PV is 500-900 clk per 128x128 score tile).  A two-pass version (maxima
// first, then exponentials) spent ~0.6 extra instructions per score plus a second chain of waits and ran 35 %
// slower regardless of head dim, so the softmax is the single-pass online form: every score is pulled out of TMEM
// and touched once.  The running maximum is kept lazily (FlashAttention-4): the reference maximum of a row only
// moves when the new chunk exceeds it by more than 2^8, so O in TMEM is rescaled (by the row's own two threads,
// between PV(j-1) and PV(j)) only a handful of times per row; P stays <= 2^8, exact in fp32 sums and safe in 16-bit
// P.  Each softmax thread pulls its half row of S into registers and hands the S buffer straight back, so the
// tensor core computes S(j+1) while the group exponentiates S(j); the two tiles ping-pong on the tensor core
// through two independent issuer warps.
// TMEM columns of tile t (base t*256): S [0,128) fp32, P [128,192) 16-bit pairs, O [192,192+dh) fp32.
#include "attn.h"
#include "launch.h"
#include "ptx.cuh"
#include "tma_util.h"

#include <algorithm>
#include <type_traits>

namespace lwb {

static constexpr int TC_BM = 128;     // query rows per CTA
static constexpr int TC_BKV = 128;    // keys per chunk
static constexpr int TC_QT = 2;                              // query tiles per CTA
static constexpr int TC_SOFT_WARPS = 8;                      // softmax warps per tile (two threads per row)
static constexpr int TC_THREADS2 = 32 * (3 + TC_QT * TC_SOFT_WARPS);   // TMA warp, 2 MMA warps, 16 softmax warps
static constexpr int TC_MMA1_WARP = 2 + TC_QT * TC_SOFT_WARPS;         // issuer warp of tile 1
static constexpr int TC_KS = 4, TC_VS = 3;                   // K / V ring depths

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
static constexpr float TC_LAZY_LOG2 = 8.f;   // the row reference maximum moves only when exceeded by more than 2^8

template <typename T, int DH>
__global__ void __launch_bounds__(TC_THREADS2, 1) attn_tc_kernel(const __grid_constant__ CUtensorMap tm, const AttnArgs p, int C) {
  constexpr int TILE_BYTES = 128 * DH * 2;                     // one 128-row tile of Q, K or V
  constexpr uint32_t PITCH = DH * 2;                           // bytes per row = swizzle span
  constexpr uint32_t LAYOUT = DH == 64 ? 2u : (DH == 32 ? 4u : 6u);   // SWIZZLE_128B / 64B / 32B
  constexpr uint32_t SBO = 8 * PITCH;                          // 8-row group stride (K-major and MN-major alike)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                          // [2] tiles
  uint8_t* sK = sQ + TC_QT * TILE_BYTES;       // [KS]
  uint8_t* sV = sK + TC_KS * TILE_BYTES;       // [VS]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + TC_VS * TILE_BYTES);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;                 // [KS]
  uint64_t* k_empty = k_full + TC_KS;          // [KS]  count = tiles in flight (one commit per MMA warp)
  uint64_t* v_full = k_empty + TC_KS;          // [VS]
  uint64_t* v_empty = v_full + TC_VS;          // [VS]
  uint64_t* s_full = v_empty + TC_VS;          // [tile]  S written by the tensor core
  uint64_t* s_free = s_full + 2;               // [tile]  every softmax warp has pulled S into registers
  uint64_t* p_full = s_free + 2;               // [tile]  P(j) written (and O rescaled if needed)
  uint64_t* p_empty = p_full + 2;              // [tile]  PV(j) has completed: P may be overwritten, O is current
  uint64_t* o_full = p_empty + 2;              // [tile]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);
  float* xch = reinterpret_cast<float*>(tmem_slot + 4);        // [parity][tile][half][128] row max / row sum exchange

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = blockIdx.y, seq = blockIdx.z;
  const int q0 = blockIdx.x * (TC_QT * TC_BM);
  const int row0 = seq * p.seqlen;                              // first matrix row of this sequence
  const int nchunks = (p.seqlen + TC_BKV - 1) / TC_BKV;
  const int ntiles = (q0 + TC_BM < p.seqlen) ? 2 : 1;           // the last CTA of a sequence may own a single tile
  const int colq = head * DH, colk = C + head * DH, colv = 2 * C + head * DH;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(q_full, 1);
    for (int i = 0; i < TC_KS; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], ntiles);
    }
    for (int i = 0; i < TC_VS; ++i) {
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], ntiles);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&s_free[t], TC_SOFT_WARPS);        // one elected arrival per softmax warp
      mbar_init(&p_full[t], TC_SOFT_WARPS);
      mbar_init(&p_empty[t], 1);
      mbar_init(&o_full[t], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_sync();   // the prologue above touched no global data; everything below reads the predecessor's output
  const int tile = warp == 1 ? 0 : (warp == TC_MMA1_WARP ? 1 : (warp - 2) / TC_SOFT_WARPS);
  const uint32_t colS = tile * 256, colP = colS + 128, colO = colS + 192;

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer
      mbar_arrive_expect_tx(q_full, ntiles * TILE_BYTES);
      for (int t = 0; t < ntiles; ++t) tma_load_2d(sQ + t * TILE_BYTES, &tm, q_full, colq, row0 + q0 + t * TC_BM);
      uint32_t kc = 0, vc = 0;
      auto load_k = [&](int j) {
        const int s = kc % TC_KS;
        mbar_wait(&k_empty[s], ((kc / TC_KS) & 1) ^ 1);
        mbar_arrive_expect_tx(&k_full[s], TILE_BYTES);
        tma_load_2d(sK + s * TILE_BYTES, &tm, &k_full[s], colk, row0 + j * TC_BKV);
        ++kc;
      };
      load_k(0);                                                 // then K(j+1) / V(j) in consumption order
      for (int j = 0; j < nchunks; ++j) {
        if (j + 1 < nchunks) load_k(j + 1);
        const int s = vc % TC_VS;
        mbar_wait(&v_empty[s], ((vc / TC_VS) & 1) ^ 1);
        mbar_arrive_expect_tx(&v_full[s], TILE_BYTES);
        tma_load_2d(sV + s * TILE_BYTES, &tm, &v_full[s], colv, row0 + j * TC_BKV);
        ++vc;
      }
    }
  } else if (warp == 1 || warp == TC_MMA1_WARP) {
    if (lane == 0 && tile < ntiles) {
      // ------------------------------------------------------------------ MMA issuer of one query tile
      constexpr bool BF = Cvt<T>::is_bf16;
      constexpr uint32_t idesc_s = umma_idesc_f16(BF, 128, TC_BKV);                    // S: N = 128 keys, both K-major
      constexpr uint32_t idesc_o = umma_idesc_f16(BF, 128, DH) | (1u << 16);           // O: B (= V) is MN-major
      uint32_t kc = 0, vc = 0;
      const uint64_t qdesc = umma_desc(smem_u32(sQ + tile * TILE_BYTES), SBO, LAYOUT);
      mbar_wait(q_full, 0);
      auto issue_s = [&]() {                                     // S(next chunk), releases the K slot
        const int s = kc % TC_KS;
        mbar_wait(&k_full[s], (kc / TC_KS) & 1);
        tc_fence_after();
        const uint64_t kdesc = umma_desc(smem_u32(sK + s * TILE_BYTES), SBO, LAYOUT);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) umma_f16_ss(tmem + colS, qdesc + 2 * kk, kdesc + 2 * kk, idesc_s, kk != 0 ? 1u : 0u);
        umma_commit(&s_full[tile]);
        umma_commit(&k_empty[s]);
        ++kc;
      };
      issue_s();
      for (int j = 0; j < nchunks; ++j) {
        if (j + 1 < nchunks) {
          mbar_wait(&s_free[tile], j & 1);                       // the group holds S(j) in registers
          issue_s();                                             // S(j+1) runs while the group exponentiates S(j)
        }
        const int vs = vc % TC_VS;
        mbar_wait(&p_full[tile], j & 1);                         // P(j) is in TMEM, O carries the current reference maximum
        mbar_wait(&v_full[vs], (vc / TC_VS) & 1);
        tc_fence_after();
        const uint64_t vdesc = umma_desc(smem_u32(sV + vs * TILE_BYTES), SBO, LAYOUT);
#pragma unroll
        for (int kk = 0; kk < TC_BKV / 16; ++kk)                 // 16 keys per MMA: A advances 8 TMEM columns, B 16 rows
          umma_f16_ts(tmem + colO, tmem + colP + 8 * kk, vdesc + ((16 * PITCH) >> 4) * kk, idesc_o, (j | kk) != 0 ? 1u : 0u);
        umma_commit(&p_empty[tile]);
        umma_commit(&v_empty[vs]);
        ++vc;
      }
      umma_commit(&o_full[tile]);
    }
  } else if (tile < ntiles) {
    // -------------------------------------------------------------------- softmax / epilogue: two threads per query row
    constexpr int OC = DH / 2;                                     // O columns owned by this thread (rescale, final store)
    static_assert(OC % 16 == 0, "the final store writes 16-column pieces");
    const int quarter = warp & 3;                                  // TMEM lane quarter this warp may access
    const int half = ((warp - 2) >> 2) & 1;                        // which 64 keys of every chunk this thread owns
    const int r = quarter * 32 + lane;
    const uint32_t tbase = tmem + (static_cast<uint32_t>(quarter * 32) << 16);
    const int xme = (tile * 2 + half) * 128 + r, xpeer = (tile * 2 + (half ^ 1)) * 128 + r;
    float m_ref = -INFINITY;                                       // reference maximum (raw scores) the exponent subtracts
    float lsum[4] = {0.f, 0.f, 0.f, 0.f};
    float v[64];
    for (int j = 0; j < nchunks; ++j) {
      // ---- pull this thread's half row of S(j) into registers and hand the S buffer back
      mbar_wait(&s_full[tile], j & 1);
      tc_fence_after();
      __syncwarp();
      tmem_ld_x32(tbase + colS + half * 64, v);
      tmem_ld_x32(tbase + colS + half * 64 + 32, v + 32);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();                                                // 32 lanes arriving on one mbarrier word serialise:
      if (lane == 0) mbar_arrive(&s_free[tile]);                   // one elected arrival per warp instead
      // ---- row maximum of the chunk: own 64 keys, then the other half's through shared memory
      const int kvalid = p.seqlen - j * TC_BKV - half * 64;        // keys >= kvalid belong to the next sequence
      float mloc;
      if (kvalid >= 64) {
        float mm[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
#pragma unroll
          for (int c = 0; c < 4; ++c) mm[c] = fmaxf(mm[c], fmaxf(v[c * 16 + i], v[c * 16 + i + 1]));
        }
        mloc = fmaxf(fmaxf(mm[0], mm[1]), fmaxf(mm[2], mm[3]));
      } else {
        mloc = -INFINITY;
#pragma unroll
        for (int i = 0; i < 64; ++i)
          if (i < kvalid) mloc = fmaxf(mloc, v[i]);
      }
      float* xb = xch + (j & 1) * 512;                             // parity double buffering: one barrier per chunk
      xb[xme] = mloc;
      named_bar_sync(1 + tile, 32 * TC_SOFT_WARPS);
      const float mchunk = fmaxf(mloc, xb[xpeer]);
      // ---- lazy reference maximum: both threads of a row take the same decision from the same numbers
      const bool move = (mchunk - m_ref) * p.scale_log2 > TC_LAZY_LOG2;   // true at j = 0 (m_ref = -inf)
      const float alpha = move ? ex2((m_ref - mchunk) * p.scale_log2) : 1.f;
      if (move) m_ref = mchunk;
      const float msc = m_ref * p.scale_log2;
#pragma unroll
      for (int i = 0; i < 4; ++i) lsum[i] *= alpha;
      // ---- P = exp2(S*scale - m_ref*scale) and the row sums, entirely in registers.  Straight-line copies (full
      // chunk / masked tail chunk) so the scheduler can interleave the sums and the packing with the exponentials.
      uint32_t pk[32];
      auto body = [&](auto tail_tag) {
        constexpr bool TAIL = decltype(tail_tag)::value;
#pragma unroll
        for (int piece = 0; piece < 2; ++piece) {
          float e[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float a = fmaf(v[piece * 32 + i], p.scale_log2, -msc);
            const float x = ex2(a);
            e[i] = (!TAIL || piece * 32 + i < kvalid) ? x : 0.f;
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            pk[piece * 16 + i] = Cvt<T>::pack(e[2 * i], e[2 * i + 1]);
            lsum[i & 3] += e[2 * i] + e[2 * i + 1];
          }
        }
      };
      if (kvalid >= 64) body(std::false_type{});
      else body(std::true_type{});
      // ---- only now wait for PV(j-1): its latency hides behind the exponentials above (P is single-buffered)
      if (j > 0) {
        mbar_wait(&p_empty[tile], (j - 1) & 1);                    // PV(j-1) done: P is free, O is complete
        tc_fence_after();
        if (__any_sync(0xffffffffu, move)) {                       // rare after the first chunks: rescale this thread's O columns
#pragma unroll
          for (int c = 0; c < OC / 8; ++c) {
            float o8[8];
            uint32_t u8[8];
            __syncwarp();
            tmem_ld_x8(tbase + colO + half * OC + c * 8, o8);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) u8[i] = __float_as_uint(o8[i] * alpha);
            tmem_st_x8(tbase + colO + half * OC + c * 8, u8);
          }
        }
      }
      __syncwarp();
      tmem_st_x16(tbase + colP + half * 32, pk);
      tmem_st_x16(tbase + colP + half * 32 + 16, pk + 16);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[tile]);
    }
    // ---- O / l -> global: the two threads of a row exchange their partial sums and each stores half of the row
    const float lpart = (lsum[0] + lsum[1]) + (lsum[2] + lsum[3]);
    float* xb = xch + (nchunks & 1) * 512;
    xb[xme] = lpart;
    named_bar_sync(1 + tile, 32 * TC_SOFT_WARPS);
    const float inv = 1.f / (lpart + xb[xpeer]);
    mbar_wait(&o_full[tile], 0);
    tc_fence_after();
    const int qrow = q0 + tile * TC_BM + r;
    T* dst = reinterpret_cast<T*>(p.o) + (static_cast<long long>(row0) + qrow) * p.ldo + head * DH + half * OC;
    __syncwarp();
#pragma unroll
    for (int c = 0; c < OC / 16; ++c) {
      float o16[16];
      __syncwarp();
      tmem_ld_x16(tbase + colO + half * OC + c * 16, o16);
      tmem_ld_wait();
      if (qrow < p.seqlen) {
        U8 o;
#pragma unroll
        for (int i = 0; i < 8; ++i) o.v[i] = Cvt<T>::pack(o16[2 * i] * inv, o16[2 * i + 1] * inv);
        stg256(dst + c * 16, o);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

template <typename T, int DH>
static int launch_tc(const AttnArgs& a, int C, cudaStream_t st) {
  CUtensorMap tm;
  std::string err;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(a.ldq), static_cast<cuuint64_t>(a.nseq) * a.seqlen};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(a.ldq) * 2};
  const cuuint32_t box[2] = {DH, 128};
  if (tma_encode(&tm, Cvt<T>::is_bf16 ? DT_BF16 : DT_F16, 2, a.q, dims, strides, box, DH * 2, &err)) return -3;
  // One CTA per SM (it allocates all 512 TMEM columns): ask for more than half of the shared memory so that a
  // second CTA can never become resident and spin inside tcgen05.alloc.
  const size_t need = 1024 + static_cast<size_t>(TC_QT + TC_KS + TC_VS) * 128 * DH * 2 + 512 + 2 * 2 * 2 * 128 * sizeof(float);
  const size_t smem = std::max<size_t>(need, 116 * 1024);
  if (int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(attn_tc_kernel<T, DH>), 200 * 1024)) return e;
  dim3 grid((a.seqlen + TC_QT * TC_BM - 1) / (TC_QT * TC_BM), a.heads, a.nseq);
  launch_k(attn_tc_kernel<T, DH>, dim3(grid), dim3(TC_THREADS2), smem, st, tm, a, C);
  return static_cast<int>(cudaGetLastError());
}

// Packed-qkv path at head dim 64: q, k, v are the column blocks [0,C), [C,2C), [2C,3C) of one 16-bit matrix.
int attention_tc_launch(int dtype, const AttnArgs& a, int dh, int C, cudaStream_t st) {
  if (dh != 64) return -2;
  return dtype == DT_BF16 ? launch_tc<__nv_bfloat16, 64>(a, C, st) : launch_tc<__half, 64>(a, C, st);
}

}  // namespace lwb
