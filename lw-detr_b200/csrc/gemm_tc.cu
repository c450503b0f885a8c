// tcgen05 / TMA GEMM family (see gemm_tc.h).  Persistent CTA PAIRS (clusters of 2, one pair per two SMs)
// compute 256 x BN output tiles with tcgen05.mma.cta_group::2 - a single-CTA tcgen05.mma was measured at about
// half of the pair rate on this part (profiles/r01c_gemm_timeline.txt), so every GEMM of the path runs paired:
//   warp 0   : TMA producer (one elected lane, in BOTH CTAs): its CTA's 128 x 64 A tile and its HALF of the
//              BN x 64 W tile per k-block, credited to the leader CTA's "full" barrier
//   warp 1   : TMEM allocator; in the leader CTA also the tcgen05.mma issuer (one lane) - accumulators are
//              double buffered in TMEM (each CTA holds its 128 rows), commits are multicast to both CTAs
//   warps 2-17: epilogue, four warps per TMEM lane quarter: tcgen05.ld -> LayerNorm-fold / bias / activation /
//              layer-scale / residual -> 16-bit (or fp32) rows to global, optional row re-ordering / pixel shuffle,
//              optional per-row (sum, sum^2) statistics for the next LayerNorm-fused GEMM.
// Replaces, on the LW-DETR path, every F.linear / nn.Conv2d / nn.ConvTranspose2d call listed in
// SURVEY.md appendix B (reference: models/backbone/vit.py:120-140,206-220, projector.py:85-132,
// transformer.py:27-39,466-517, ops/modules/ms_deform_attn.py:112-143, lwdetr.py:149-159).
#include "gemm_tc.h"
#include "launch.h"
#include "ptx.cuh"
#include "tma_util.h"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace lwb {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int A_STAGE_BYTES = BM * BK * 2;
static constexpr int EPI_WARPS = 16;                      // two groups of 8 (alternate tiles); in a group two warps per TMEM lane quarter, half of the columns each
static constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS;
static constexpr int MAX_STAGES = 8;

// Exact (erf) GELU, nn.GELU() default used by timm's Mlp (vit.py:184).  gelu(x) = x*Phi(x) with
// Phi(-|x|) = 0.5*erfc(|x|/sqrt2) from Abramowitz-Stegun 7.1.26 (|erf error| <= 1.5e-7):
//   gelu(x) = max(x, 0) - |x| * [0.5 * poly(t) * exp(-x^2/2)],  t = 1 / (1 + p|x|/sqrt2)
// 14 instructions incl. 2 MUFU instead of ~30 for erff(); max abs deviation from the erff form 2.2e-7.
__device__ __forceinline__ float gelu_erf(float x) {
  const float ax = fabsf(x);
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.2316418882f, ax, 1.0f)));       // 0.3275911 / sqrt(2)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752044448170f));        // exp(-x^2/2)
  float p = fmaf(0.5307027145f, t, -0.7265760135f);                                          // 0.5 * A&S coefficients
  p = fmaf(p, t, 0.7107068705f);
  p = fmaf(p, t, -0.142248368f);
  p = fmaf(p, t, 0.127414796f);
  return fmaf(-ax * t, p * e, fmaxf(x, 0.f));
}

// The same exact-erf GELU for a PAIR on the packed fp32x2 pipe, without the MUFU: gelu(x) = x * (0.5 + xc * q(xc^2)), xc = x
// clamped to [-4.5, 4.5], q a degree-9 polynomial fitted to erf(x/sqrt2) / (2x) (weighted least squares at Chebyshev nodes;
// fp32 Horner: max |error| 7.4e-5 at |x| ~ 4.46 where gelu ~ 4.46, < 1e-5 for |x| < 3 (tests/test_numerics_cpu.py); beyond the clamp Phi(-4.5) = 3.4e-6
// multiplies x).  16 instructions per pair (8 per element) against 14 per element for gelu_erf - the fc1 epilogue is bound by
// its instruction count, not by the tensor core (DESIGN.md section 3).
__device__ __forceinline__ uint64_t gelu_erf2(uint64_t x2) {
  float x0, x1;
  f2_unpack(x2, x0, x1);
  const uint64_t xc = f2_pack(fminf(fmaxf(x0, -4.5f), 4.5f), fminf(fmaxf(x1, -4.5f), 4.5f));
  const uint64_t u = f2_mul(xc, xc);
#define LWB_K2(v) f2_pack(v, v)
  uint64_t q = f2_fma(LWB_K2(-1.3369040159e-12f), u, LWB_K2(1.6336444415e-10f));
  q = f2_fma(q, u, LWB_K2(-8.9213697499e-09f));
  q = f2_fma(q, u, LWB_K2(2.8944761772e-07f));
  q = f2_fma(q, u, LWB_K2(-6.2733902842e-06f));
  q = f2_fma(q, u, LWB_K2(9.7063541348e-05f));
  q = f2_fma(q, u, LWB_K2(-1.1183810776e-03f));
  q = f2_fma(q, u, LWB_K2(9.8202145566e-03f));
  q = f2_fma(q, u, LWB_K2(-6.6317755718e-02f));
  q = f2_fma(q, u, LWB_K2(3.9887377948e-01f));
  const uint64_t t = f2_fma(xc, q, LWB_K2(0.5f));
#undef LWB_K2
  return f2_mul(x2, t);
}

struct TileCoord {
  int m_tile, n_tile, n0, cb, cy0, cx0;
};
// pair-tile index -> this CTA's (m_tile, n_tile); n fastest, so neighbouring pairs share the A rows in L2
__device__ __forceinline__ TileCoord decode_tile(const GemmArgs& p, int ptile, int rank, int BN) {
  TileCoord t;
  t.n_tile = ptile % p.n_tiles;
  t.m_tile = 2 * (ptile / p.n_tiles) + rank;     // may be == m_tiles for the odd tail: loads are OOB zero-fill, stores masked
  t.n0 = t.n_tile * BN;
  t.cb = t.cy0 = t.cx0 = 0;
  if (p.a_mode != AMODE_PLAIN) {
    const int per_img = p.tiles_x * p.tiles_y;
    t.cb = t.m_tile / per_img;                    // == batch for the odd tail: out of bounds in the TMA batch dimension
    const int r = t.m_tile % per_img;
    t.cy0 = (r / p.tiles_x) * p.TH;
    t.cx0 = (r % p.tiles_x) * p.TW;
  }
  return t;
}

// Persistent CTA pairs: pair q (= blockIdx.x / 2) walks pair-tiles q, q + npairs, ...  A pair-tile is two
// vertically adjacent 128-row m-tiles (CTA rank 0 / 1) times one BN-wide n-tile.  The smem ring (TMA -> MMA)
// runs continuously across tiles and the accumulator is double buffered in TMEM, so the epilogue of tile i
// overlaps the loads and MMAs of tile i+1.
// EP (epilogue specialisation): EP_GENERIC keeps every feature behind runtime flags; the others compile the
// features of the hot GEMMs in or out so the per-element instruction count stays minimal:
//   EP_BIAS      out = acc + bias                     (16-bit out, plain rows, no LN / residual / activation)
//   EP_BIAS_ACT  out = act(acc + bias)                (activation still a runtime switch, hoisted per chunk)
//   EP_LN        out = LN-fold(acc) + bias            (qkv)
//   EP_LN_GELU   out = gelu(LN-fold(acc) + bias)      (fc1)
//   EP_RESID     out = resid + gamma*(acc + bias), optional row statistics (proj, fc2, patch embed, decoder)
enum : int { EP_GENERIC = 0, EP_BIAS = 1, EP_BIAS_ACT = 2, EP_LN = 3, EP_LN_GELU = 4, EP_RESID = 5 };

__device__ __forceinline__ float4 lds128(const float* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
  return v;
}

template <typename T, int BN, int EP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs p) {
  constexpr int B_HALF_BYTES = (BN / 2) * BK * 2;                             // this CTA's half of the W tile
  constexpr uint32_t ACC_STRIDE = BN <= 64 ? 64 : (BN <= 128 ? 128 : 256);   // TMEM columns per accumulator buffer
  constexpr uint32_t TMEM_COLS = 2 * ACC_STRIDE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stages = p.stages;
  uint8_t* sA = smem;
  uint8_t* sB = smem + stages * A_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + stages * B_HALF_BYTES);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* acc_full = empty_bar + MAX_STAGES;      // [2]
  uint64_t* acc_empty = acc_full + 2;               // [2]  (used in the leader CTA)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* s_vec = reinterpret_cast<float*>(full_bar + 32);   // 256 B of barriers, then {bias | gamma | colsum}[n_tiles * BN]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();          // 0 = leader
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int m_pairs = (p.m_tiles + 1) >> 1;
  const int num_ptiles = m_pairs * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 2);                   // leader: own arrive.expect_tx + the peer's remote arrive
      mbar_init(&empty_bar[s], 1);                  // one multicast tcgen05.commit
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], p.epi_groups == 2 ? EPI_WARPS : 2 * EPI_WARPS);   // the epilogue warps (of one group / of both) in each of the two CTAs
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_slot, TMEM_COLS);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync_all();                               // barriers of BOTH CTAs are initialised before any remote use
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();   // the prologue above touched no global data; everything below reads the predecessor's output

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer (both CTAs)
      uint32_t ring = 0;
      for (int pt = pair; pt < num_ptiles; pt += npairs) {
        const TileCoord tc = decode_tile(p, pt, static_cast<int>(rank), BN);
        for (int kb = 0; kb < p.kblocks; ++kb, ++ring) {
          const int s = ring % stages;
          const uint32_t ph = (ring / stages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* a_dst = sA + s * A_STAGE_BYTES;
          if (p.a_mode == AMODE_PLAIN) {
            tma2_load_2d(a_dst, &tmA, &full_bar[s], kb * BK, tc.m_tile * BM);
          } else {
            const int tap = kb / p.cin_blocks;
            const int c0 = (kb % p.cin_blocks) * BK;
            const int dy = tap / 3, dx = tap % 3;
            if (p.a_mode == AMODE_CONV3_S1) {
              tma2_load_4d(a_dst, &tmA, &full_bar[s], c0, tc.cx0 + dx - 1, tc.cy0 + dy - 1, tc.cb);
            } else {
              // input row iy = 2*oy + dy - 1 = 2*(oy + yoff) + py ; same for columns
              const int py = (dy == 1) ? 0 : 1, yoff = (dy == 0) ? -1 : 0;
              const int px = (dx == 1) ? 0 : 1, xoff = (dx == 0) ? -1 : 0;
              tma2_load_5d(a_dst, &tmA, &full_bar[s], px * p.lda + c0, tc.cx0 + xoff, py, tc.cy0 + yoff, tc.cb);
            }
          }
          tma2_load_2d(sB + s * B_HALF_BYTES, &tmB, &full_bar[s], kb * BK, tc.n0 + static_cast<int>(rank) * (BN / 2));
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[s], 2u * (p.a_stage_tx + B_HALF_BYTES));
          else mbar_arrive_cluster(&full_bar[s], 0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      // ------------------------------------------------------------------ MMA issuer (leader CTA only)
      constexpr uint32_t idesc = umma_idesc_f16(Cvt<T>::is_bf16, 2 * BM, BN);
      uint32_t ring = 0;
      int it = 0;
      for (int pt = pair; pt < num_ptiles; pt += npairs, ++it) {
        const int buf = it & 1;
        mbar_wait(&acc_empty[buf], ((it >> 1) & 1) ^ 1);     // both epilogues have drained this accumulator buffer
        tc_fence_after();
        const uint32_t tacc = tmem_base + buf * ACC_STRIDE;
        for (int kb = 0; kb < p.kblocks; ++kb, ++ring) {
          const int s = ring % stages;
          const uint32_t ph = (ring / stages) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint64_t adesc = umma_desc_k128(smem_u32(sA + s * A_STAGE_BYTES));
          const uint64_t bdesc = umma_desc_k128(smem_u32(sB + s * B_HALF_BYTES));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 elements (32 B) along K inside the 128 B swizzle row: +2 in 16-byte units
            umma2_f16_ss(tacc, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma2_commit_both(&empty_bar[s]);                   // frees the stage in both CTAs
        }
        umma2_commit_both(&acc_full[buf]);
      }
    }
  } else {
    // -------------------------------------------------------------------- epilogue (16 warps, both CTAs)
    const int quarter = warp & 3;               // TMEM lanes [32*quarter, 32*quarter+32) (hardware: warp_id % 4)
    // The 16 epilogue warps form TWO GROUPS.  With many tiles per CTA (epi_groups = 2: qkv, fc1, ...) the groups take alternate
    // tiles (group g owns accumulator buffer g): while one group is in the latency-bound head of its tile (statistics, TMEM
    // pull, residual) or in its stores, the other one is in its arithmetic - as one group the four warps of a scheduler moved in
    // lock step and left the FMA pipe idle half of the time (fc1: FMA pipe 52 % busy at an FMA-bound epilogue,
    // profiles/r02_ncu_gemm_small.txt).  Measured in the small / B = 32 step: qkv 257 -> 233 us, fc1 364 -> 353 us per 10
    // launches.  With two or three tiles per CTA (proj, fc2, the projector) halving the warps per tile only stretches the tail
    // (fc2 274 -> 309 us), so there both groups split every tile (epi_groups = 1: group g takes half of the pull rounds).
    const int grp = (warp - 2) >> 3;
    const int chalf = ((warp - 2) >> 2) & 1;    // which half of the tile's 16-column chunks this warp owns
    const int r = quarter * 32 + lane;          // row inside this CTA's 128-row tile
    constexpr bool GEN = EP == EP_GENERIC;
    const bool has_gamma = (GEN || EP == EP_RESID) && p.gamma != nullptr;
    const bool ln_in = GEN ? (p.stats_in != nullptr) : (EP == EP_LN || EP == EP_LN_GELU);
    const int act = GEN || EP == EP_BIAS_ACT ? p.act : (EP == EP_LN_GELU ? ACT_GELU : ACT_NONE);
    const bool has_resid = (GEN || EP == EP_RESID) && p.resid != nullptr;
    const bool do_stats = (GEN || EP == EP_RESID) && p.stats_out != nullptr;
    const bool plain_out = !GEN;                 // 16-bit, rows in place, no pixel shuffle
    // Stage the bias / layer-scale / LayerNorm column-sum vectors of ALL n-tiles once per CTA (epilogue warps only,
    // while the producer / MMA warps already stream the first tile): the per-tile epilogue then has no dependent
    // global loads except the (prefetched) residual and the per-row LayerNorm statistics.
    {
      const int npad_all = p.n_tiles * BN;
      for (int i = threadIdx.x - 64; i < npad_all; i += 32 * EPI_WARPS) {
        const bool in = i < p.N;
        s_vec[i] = (p.bias != nullptr && in) ? __ldg(p.bias + i) : 0.f;
        s_vec[npad_all + i] = (p.gamma != nullptr && in) ? __ldg(p.gamma + i) : 1.f;
        s_vec[2 * npad_all + i] = (p.colsum != nullptr && in) ? __ldg(p.colsum + i) : 0.f;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
    }
    int it = 0;
    const int n_my_tiles = pair < num_ptiles ? (num_ptiles - pair + npairs - 1) / npairs : 0;
    // Tile walk without a division per tile (plain GEMMs; ncu counted ~180 of the 324 instructions a warp spends per qkv tile
    // in tile decoding, row bookkeeping and the statistics reduction - more than on its 48 output columns): pair-tile index
    // pt = m_pair * n_tiles + n_tile advances by npairs = d_mp * n_tiles + d_nt with a carry.
    const bool plain = p.a_mode == AMODE_PLAIN;
    const bool alt = p.epi_groups == 2;
    const int tstep = alt ? 2 * npairs : npairs;        // this group's next tile
    const int d_mp = tstep / p.n_tiles, d_nt = tstep - d_mp * p.n_tiles;
    const int pt0 = alt ? pair + grp * npairs : pair;
    int w_nt = pt0 % p.n_tiles, w_mp = pt0 / p.n_tiles;
    auto plain_tile = [&](int nt, int mp) {
      TileCoord t;
      t.n_tile = nt;
      t.m_tile = 2 * mp + static_cast<int>(rank);
      t.n0 = nt * BN;
      t.cb = t.cy0 = t.cx0 = 0;
      return t;
    };
    // LayerNorm statistics of a row: the producer's partial (sum, sum of squares) pairs.  The partials of the NEXT tile's rows
    // are requested at the start of a tile and reduced at its end (first four in registers), so the L2 round trip that used to
    // stall the first use (13 % of all samples of the qkv GEMM on one FADD) overlaps the tile's own work.
    float nx_mean = 0.f, nx_rstd = 1.f;
    // combine equal-width partials (sum_p, M2_p): mean = sum(sum_p) / C, var = [sum(M2_p) + n_p * sum((sum_p / n_p - mean)^2)] / C
    const float part_n = p.stats_parts_in > 0 ? 1.f / (p.ln_inv_c * p.stats_parts_in) : 1.f, part_inv_n = 1.f / part_n;
    auto stats_of = [&](long long mrow, float& mean, float& rstd) {
      float s1 = 0.f, m2 = 0.f;
      for (int i = 0; i < p.stats_parts_in; ++i) s1 += __ldg(p.stats_in + mrow * p.stats_parts_in + i).x;
      mean = s1 * p.ln_inv_c;
      for (int i = 0; i < p.stats_parts_in; ++i) {
        const float2 q = __ldg(p.stats_in + mrow * p.stats_parts_in + i);
        const float dm = q.x * part_inv_n - mean;
        m2 += q.y + part_n * dm * dm;
      }
      rstd = rsqrtf(m2 * p.ln_inv_c + p.ln_eps);
    };
    if (ln_in && plain && pt0 < num_ptiles) {
      const long long m0 = static_cast<long long>(2 * w_mp + static_cast<int>(rank)) * BM + r;
      if (m0 < p.M) stats_of(m0, nx_mean, nx_rstd);
    }
    it = alt ? grp : 0;
    const int it_step = alt ? 2 : 1;
    for (int pt = pt0; pt < num_ptiles; pt += tstep, it += it_step) {
      const TileCoord tc = plain ? plain_tile(w_nt, w_mp) : decode_tile(p, pt, static_cast<int>(rank), BN);
      // next tile of this group
      w_nt += d_nt;
      w_mp += d_mp;
      if (w_nt >= p.n_tiles) {
        w_nt -= p.n_tiles;
        ++w_mp;
      }
      const int n0 = tc.n0;
      const int buf = it & 1;
      int m, b = 0, y = 0, x = 0;
      bool valid;
      if (p.a_mode == AMODE_PLAIN) {
        m = tc.m_tile * BM + r;
        valid = m < p.M;
        if (GEN && (p.remap_rows || p.shuffle_cout)) {
          const int per = p.IH * p.IW;
          b = m / per;
          const int rem = m - b * per;
          if (p.rows_in == ROWS_WINDOW_MAJOR) {
            const int wh = p.IH >> 2, ww = p.IW >> 2, wsz = wh * ww;
            const int win = rem / wsz, t = rem - win * wsz;
            y = (win >> 2) * wh + t / ww;
            x = (win & 3) * ww + t % ww;
          } else {
            y = rem / p.IW;
            x = rem - y * p.IW;
          }
        }
      } else {
        const int ry = r / p.TW;
        y = tc.cy0 + ry;
        x = tc.cx0 + (r - ry * p.TW);
        b = tc.cb;
        valid = (tc.m_tile < p.m_tiles) && (r < p.TW * p.TH) && (y < p.OH) && (x < p.OW);
        m = (b * p.OH + y) * p.OW + x;
      }
      long long out_row = m;
      if (GEN && p.remap_rows) out_row = (static_cast<long long>(b) * p.IH + y) * p.IW + x;
      const long long res_row = p.resid_mod > 0 ? (m % p.resid_mod) : m;
      const bool zero_row = GEN && p.row_zero != nullptr && valid && __ldg(p.row_zero + m) != 0;

      const int npad = p.n_tiles * BN;
      const float* s_bias = s_vec + n0;
      const float* s_gamma = s_vec + npad + n0;
      const float* s_csum = s_vec + 2 * npad + n0;
      // fused LayerNorm (consumer): combine the producer's partial sums of this row
      float ln_mean = 0.f, ln_rstd = 1.f;
      float2 nq[4];
      long long nx_row = -1;
      if (ln_in && plain) {
        ln_mean = nx_mean;                            // reduced at the end of the previous tile (or before the loop)
        ln_rstd = nx_rstd;
        if (pt + tstep < num_ptiles) {
          const long long mn = static_cast<long long>(2 * w_mp + static_cast<int>(rank)) * BM + r;
          if (mn < p.M) {
            nx_row = mn;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < p.stats_parts_in) nq[i] = __ldg(p.stats_in + mn * p.stats_parts_in + i);
          }
        }
      } else if (ln_in && valid) {
        stats_of(m, ln_mean, ln_rstd);
      }
      // Row statistics for the fused LayerNorm of the consumer, SHIFTED by the first value of the slice: sums of (x - K) and
      // (x - K)^2 do not cancel when the row mean is large against its spread (real checkpoints; E[x^2] - mean^2 would).
      float st_sum = 0.f, st_sq = 0.f, st_K = 0.f;
      bool st_have = false;
      int st_n = 0;
      const T* resid_row = has_resid ? reinterpret_cast<const T*>(p.resid) + res_row * p.ld_resid : nullptr;

      // one 16-column chunk: LN-fold / bias / activation / layer-scale / residual / store
      auto finish_chunk = [&](int c, float (&v)[16], const U8& rr, bool rvec) {
        const int n = n0 + c * 16;
        const int nrem = p.N - n;                     // may be <= 0 for the padded tail of the last n-tile
        if (!valid || nrem <= 0) return;
        const bool full = nrem >= 16;
        // packed fp32x2 from here on (FFMA2 / FADD2 / FMUL2): half the issue slots of the scalar form
        uint64_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = f2_pack(v[2 * j], v[2 * j + 1]);
        {
          const float4* sb = reinterpret_cast<const float4*>(s_bias + c * 16);
          if (ln_in) {
            // rstd*(acc - mean*colsum) + bias  ==  a*acc + (b*colsum + bias),  a = rstd, b = -rstd*mean
            const uint64_t a2 = f2_pack(ln_rstd, ln_rstd), b2 = f2_pack(-ln_rstd * ln_mean, -ln_rstd * ln_mean);
            const float4* sc = reinterpret_cast<const float4*>(s_csum + c * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 c4 = lds128(reinterpret_cast<const float*>(sc + j));
              const float4 b4 = lds128(reinterpret_cast<const float*>(sb + j));
              w[2 * j] = f2_fma(a2, w[2 * j], f2_fma(b2, f2_pack(c4.x, c4.y), f2_pack(b4.x, b4.y)));
              w[2 * j + 1] = f2_fma(a2, w[2 * j + 1], f2_fma(b2, f2_pack(c4.z, c4.w), f2_pack(b4.z, b4.w)));
            }
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b4 = lds128(reinterpret_cast<const float*>(sb + j));
              w[2 * j] = f2_add(w[2 * j], f2_pack(b4.x, b4.y));
              w[2 * j + 1] = f2_add(w[2 * j + 1], f2_pack(b4.z, b4.w));
            }
          }
        }
        if (act == ACT_GELU) {
#pragma unroll
          for (int j = 0; j < 8; ++j) w[j] = gelu_erf2(w[j]);
        } else if (act == ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float a, b;
            f2_unpack(w[j], a, b);
            w[j] = f2_pack(fmaxf(a, 0.f), fmaxf(b, 0.f));
          }
        } else if (act == ACT_SILU) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float a, b;
            f2_unpack(w[j], a, b);
            w[j] = f2_pack(__fdividef(a, 1.f + __expf(-a)), __fdividef(b, 1.f + __expf(-b)));
          }
        }
        if (has_gamma) {
          const float4* sg = reinterpret_cast<const float4*>(s_gamma + c * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 g4 = lds128(reinterpret_cast<const float*>(sg + j));
            w[2 * j] = f2_mul(w[2 * j], f2_pack(g4.x, g4.y));
            w[2 * j + 1] = f2_mul(w[2 * j + 1], f2_pack(g4.z, g4.w));
          }
        }
        if (rvec) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 f = Cvt<T>::unpack(rr.v[j]);
            w[j] = f2_add(w[j], f2_pack(f.x, f.y));
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) f2_unpack(w[j], v[2 * j], v[2 * j + 1]);
        if (!rvec && (GEN || EP == EP_RESID) && resid_row != nullptr) {
          for (int j = 0; j < 16; ++j)
            if (j < nrem) v[j] += Cvt<T>::to_f(resid_row[n + j]);
        }
        if (GEN && zero_row) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
        }
        // destination
        long long orow = out_row;
        int ocol = n;
        if (GEN && p.hm_S > 0) {                      // head-major: one 16-column chunk = one (slice, head), ld_out == 16
          const int dd = p.hm_heads * 16;
          const int slice = n / dd, head = (n - slice * dd) >> 4;
          const int bb = m / p.hm_S, ss = m - bb * p.hm_S;
          orow = ((static_cast<long long>(bb) * p.hm_slices + slice) * p.hm_heads + head) * p.hm_S + ss;
          ocol = 0;
        }
        if (GEN && p.shuffle_cout > 0) {
          const int q = n / p.shuffle_cout;
          ocol = n - q * p.shuffle_cout;
          orow = (static_cast<long long>(b) * (2 * p.IH) + 2 * y + (q >> 1)) * (2 * p.IW) + 2 * x + (q & 1);
        }
        if (!plain_out && p.out_fp32) {
          float* op = reinterpret_cast<float*>(p.out) + orow * p.ld_out + ocol;
          if (full && (reinterpret_cast<uintptr_t>(op) & 15) == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              reinterpret_cast<float4*>(op)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
            for (int j = 0; j < 16; ++j)
              if (j < nrem) op[j] = v[j];
          }
        } else {
          T* op = reinterpret_cast<T*>(p.out) + orow * p.ld_out + ocol;
          if (full && (reinterpret_cast<uintptr_t>(op) & 31) == 0) {
            U8 o;
#pragma unroll
            for (int j = 0; j < 8; ++j) o.v[j] = Cvt<T>::pack(v[2 * j], v[2 * j + 1]);
            stg256(op, o);
            if (do_stats) {                           // statistics of the ROUNDED values the consumer will read
              st_n += 16;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float2 f = Cvt<T>::unpack(o.v[j]);
                if (!st_have) {
                  st_K = f.x;
                  st_have = true;
                }
                const float d0 = f.x - st_K, d1 = f.y - st_K;
                st_sum += d0 + d1;
                st_sq = fmaf(d0, d0, fmaf(d1, d1, st_sq));
              }
            }
          } else {
            for (int j = 0; j < 16; ++j)
              if (j < nrem) {
                const T h = Cvt<T>::from_f(v[j]);
                op[j] = h;
                if (do_stats) {
                  const float f = Cvt<T>::to_f(h);
                  if (!st_have) {
                    st_K = f;
                    st_have = true;
                  }
                  const float d0 = f - st_K;
                  ++st_n;
                  st_sum += d0;
                  st_sq = fmaf(d0, d0, st_sq);
                }
              }
          }
        }
      };
      // residual prefetch for a chunk (independent of the accumulator)
      auto resid_prefetch = [&](int c, U8& rr) -> bool {
        const int n = n0 + c * 16;
        if ((GEN || EP == EP_RESID) && valid && (p.N - n) >= 16 && resid_row != nullptr && (reinterpret_cast<uintptr_t>(resid_row + n) & 31) == 0) {
          rr = ldg256(resid_row + n);
          return true;
        }
        return false;
      };

      constexpr int CH_PER_WARP = BN / 16 / 2;
      // The slice is pulled G chunks (16 columns each) at a time - the kernel runs at 96 registers per thread - and the TMEM
      // buffer goes back to the MMA warp right after this warp's LAST pull, before that round's math / stores.
      constexpr int G = CH_PER_WARP % 3 == 0 ? 3 : (CH_PER_WARP >= 4 ? 2 : 1);
      constexpr int NR = CH_PER_WARP / G;               // pull rounds per column half: 4 / 2 / 2 / 2 for BN = 256 / 192 / 128 / 64
      static_assert(CH_PER_WARP % G == 0 && NR % 2 == 0, "chunk rounds");
      const int rd0 = alt ? 0 : grp * (NR / 2), rd1 = alt ? NR : rd0 + NR / 2;   // this warp's rounds
      const int c_first = chalf * CH_PER_WARP;
      U8 rr_cur, rr_nxt;
      bool rv_cur = resid_prefetch(c_first + rd0 * G, rr_cur), rv_nxt = false;

      mbar_wait(&acc_full[buf], (it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr_row = tmem_base + buf * ACC_STRIDE + (static_cast<uint32_t>(quarter * 32) << 16);
      float v[G][16];
#pragma unroll 1                                    // one copy of the (large) chunk code: the rounds differ only in their column offset
      for (int rd = rd0; rd < rd1; ++rd) {
        __syncwarp();                                 // tcgen05.ld is .sync.aligned: reconverge first
#pragma unroll
        for (int i = 0; i < G; ++i) tmem_ld_x16(taddr_row + (c_first + rd * G + i) * 16, v[i]);
        tmem_ld_wait();
        if (rd == rd1 - 1) {
          tc_fence_before();
          __syncwarp();
          // (the release of the last two tiles is never consumed: skipping it also guarantees that no remote arrive is
          //  still in flight when the pair leaves through the relaxed cluster rendezvous below)
          if (lane == 0 && it + 2 < n_my_tiles) {
            if (rank == 0) mbar_arrive(&acc_empty[buf]);
            else mbar_arrive_cluster(&acc_empty[buf], 0);
          }
        }
#pragma unroll
        for (int i = 0; i < G; ++i) {
          const int c = rd * G + i;
          if (c + 1 < rd1 * G) rv_nxt = resid_prefetch(c_first + c + 1, rr_nxt);
          finish_chunk(c_first + c, v[i], rr_cur, rv_cur);
          rr_cur = rr_nxt;
          rv_cur = rv_nxt;
        }
      }
      if (do_stats && valid) {
        // partial = (sum of the slice, sum of squared deviations from the slice's own mean); every slice has the same width
        // (gemm_build checks N % BN == 0 for producers), which is all the consumer needs to combine them (Chan et al.)
        const float nn = static_cast<float>(st_n > 0 ? st_n : 1);
        const float part_sum = fmaf(nn, st_K, st_sum), part_m2 = fmaxf(st_sq - st_sum * st_sum / nn, 0.f);
        p.stats_out[static_cast<long long>(m) * p.stats_parts_out + (alt ? tc.n_tile * 2 + chalf : tc.n_tile * 4 + chalf * 2 + grp)] = make_float2(part_sum, part_m2);
      }
      if (nx_row >= 0) {                              // statistics of the next tile's row: the requests above have landed by now
        float s1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (i < p.stats_parts_in) s1 += nq[i].x;
        for (int i = 4; i < p.stats_parts_in; ++i) s1 += __ldg(p.stats_in + nx_row * p.stats_parts_in + i).x;
        nx_mean = s1 * p.ln_inv_c;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (i < p.stats_parts_in) {
            const float dm = nq[i].x * part_inv_n - nx_mean;
            m2 += nq[i].y + part_n * dm * dm;
          }
        for (int i = 4; i < p.stats_parts_in; ++i) {
          const float2 q = __ldg(p.stats_in + nx_row * p.stats_parts_in + i);
          const float dm = q.x * part_inv_n - nx_mean;
          m2 += q.y + part_n * dm * dm;
        }
        nx_rstd = rsqrtf(m2 * p.ln_inv_c + p.ln_eps);
      }
    }
  }

  tc_fence_before();
  cluster_sync_relaxed();                           // nobody frees TMEM / exits while its peer may still use it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------- host
static int encode(CUtensorMap* tm, int dtype, int rank, const void* base, const cuuint64_t* dims,
                  const cuuint64_t* strides_bytes, const cuuint32_t* box, std::string* err) {
  return tma_encode(tm, dtype, rank, base, dims, strides_bytes, box, 128, err);
}

static int num_sms() { return current_device_sms(); }

static int pick_bn(int N, int m_tiles) {
  int bn;
  if (N <= 64) bn = 64;
  else if (N <= 128) bn = 128;
  else {
    const int cand[3] = {256, 192, 128};
    int best = 256, best_waste = 1 << 30;
    for (int c : cand) {
      const int waste = ((N + c - 1) / c) * c - N;
      if (waste < best_waste) { best_waste = waste; best = c; }
    }
    bn = best;
  }
  // Small problems: prefer more CTAs over wider tiles so that all 148 SMs get work.
  auto tiles = [&](int b) { return static_cast<long long>((m_tiles + 1) / 2) * ((N + b - 1) / b); };
  while (bn > 64 && tiles(bn) < 74) {
    const int nb = bn == 256 ? 128 : (bn == 192 ? 64 : 64);
    if (((N + nb - 1) / nb) * nb - N > ((N + bn - 1) / bn) * bn - N + 32) break;
    bn = nb;
  }
  return bn;
}

int gemm_build(const GemmDesc& d, GemmOp* op, std::string* err) {
  std::memset(op, 0, sizeof(*op));
  if (d.K % BK != 0 || d.K <= 0) { *err = "gemm: K must be a positive multiple of 64"; return -1; }
  if (!d.out_fp32 && (d.ld_out % 8) != 0) { *err = "gemm: 16-bit ld_out must be a multiple of 8"; return -1; }
  if ((d.lda % 8) != 0) { *err = "gemm: lda must be a multiple of 8"; return -1; }
  GemmArgs& a = op->args;
  a.M = d.M; a.N = d.N; a.kblocks = d.K / BK; a.a_mode = d.a_mode; a.lda = d.lda;
  a.bias = d.bias; a.gamma = d.gamma; a.resid = d.resid; a.ld_resid = d.ld_resid; a.resid_mod = d.resid_mod;
  a.act = d.act; a.out = d.out; a.ld_out = d.ld_out; a.out_fp32 = d.out_fp32;
  a.rows_in = d.rows_in; a.remap_rows = d.remap_rows; a.shuffle_cout = d.shuffle_cout; a.IH = d.IH; a.IW = d.IW;
  a.hm_S = d.hm_S; a.hm_heads = d.hm_heads; a.hm_slices = d.hm_slices; a.row_zero = d.row_zero;
  if (d.hm_S > 0) {
    if (d.a_mode != AMODE_PLAIN || d.remap_rows || d.shuffle_cout || d.out_fp32 || d.hm_heads < 1 || d.hm_slices < 1 ||
        d.N != d.hm_slices * d.hm_heads * 16 || d.M % d.hm_S != 0) { *err = "gemm: head-major store needs a plain 16-bit GEMM with N == slices*heads*16 and M % S == 0"; return -1; }
    a.ld_out = 16;
  }
  if (d.out_fp32 && d.ld_out < d.N) { *err = "gemm: fp32 ld_out must be >= N"; return -1; }
  a.stats_out = d.stats_out; a.stats_in = d.stats_in; a.stats_parts_in = d.stats_parts_in; a.colsum = d.colsum;
  a.ln_inv_c = d.ln_C > 0 ? 1.f / d.ln_C : 0.f; a.ln_eps = d.ln_eps;
  if ((d.stats_out || d.stats_in) && (d.a_mode != AMODE_PLAIN || d.remap_rows || d.shuffle_cout || d.out_fp32)) { *err = "gemm: LN fusion needs a plain 16-bit GEMM"; return -1; }
  if (d.stats_in && (!d.colsum || d.stats_parts_in <= 0 || d.ln_C <= 0 || d.ln_C % d.stats_parts_in != 0)) { *err = "gemm: LN consumer needs colsum / parts / C (C a multiple of the partial count)"; return -1; }
  op->dtype = d.dtype;
  if ((d.remap_rows || d.shuffle_cout) && (d.IH <= 0 || d.IW <= 0 || d.M % (d.IH * d.IW) != 0)) {
    *err = "gemm: row remap needs IH/IW with M a multiple of IH*IW"; return -1;
  }
  if (d.rows_in == ROWS_WINDOW_MAJOR && ((d.IH % 4) || (d.IW % 4))) { *err = "gemm: window grid needs IH,IW % 4 == 0"; return -1; }
  if (d.shuffle_cout > 0 && (d.shuffle_cout % 16 != 0 || d.N != 4 * d.shuffle_cout)) {
    *err = "gemm: pixel-shuffle needs N == 4*cout, cout % 16 == 0"; return -1;
  }

  int m_tiles;
  if (d.a_mode == AMODE_PLAIN) {
    m_tiles = (d.M + BM - 1) / BM;
    a.a_stage_tx = A_STAGE_BYTES;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(d.K), static_cast<cuuint64_t>(d.M)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(d.lda) * 2};
    const cuuint32_t box[2] = {BK, BM};
    if (encode(&op->ta, d.dtype, 2, d.A, dims, strides, box, err)) return -1;
  } else {
    if (d.K % 9 != 0 || (d.K / 9) % BK != 0) { *err = "gemm: conv needs K = 9*Cin, Cin % 64 == 0"; return -1; }
    if (d.M != d.B * d.OH * d.OW) { *err = "gemm: conv needs M == B*OH*OW"; return -1; }
    const int cin = d.K / 9;
    a.cin_blocks = cin / BK;
    a.OH = d.OH; a.OW = d.OW;
    // tile = TW x TH output pixels (<= 128): maximise useful rows
    int best_tw = 1, best_th = 1; double best_u = -1;
    for (int tw = 1; tw <= std::min(d.OW, 128); ++tw) {
      const int th = std::min(128 / tw, d.OH);
      const long long tiles = static_cast<long long>((d.OW + tw - 1) / tw) * ((d.OH + th - 1) / th);
      const double u = static_cast<double>(d.OW) * d.OH / (tiles * 128.0);
      if (u > best_u + 1e-9) { best_u = u; best_tw = tw; best_th = th; }
    }
    a.TW = best_tw; a.TH = best_th;
    a.tiles_x = (d.OW + a.TW - 1) / a.TW;
    a.tiles_y = (d.OH + a.TH - 1) / a.TH;
    m_tiles = d.B * a.tiles_x * a.tiles_y;
    a.a_stage_tx = static_cast<uint32_t>(a.TW * a.TH * BK * 2);
    if (d.a_mode == AMODE_CONV3_S1) {
      const cuuint64_t dims[4] = {static_cast<cuuint64_t>(cin), static_cast<cuuint64_t>(d.OW),
                                  static_cast<cuuint64_t>(d.OH), static_cast<cuuint64_t>(d.B)};
      const cuuint64_t strides[3] = {static_cast<cuuint64_t>(d.lda) * 2, static_cast<cuuint64_t>(d.OW) * d.lda * 2,
                                     static_cast<cuuint64_t>(d.OH) * d.OW * d.lda * 2};
      const cuuint32_t box[4] = {BK, static_cast<cuuint32_t>(a.TW), static_cast<cuuint32_t>(a.TH), 1};
      if (encode(&op->ta, d.dtype, 4, d.A, dims, strides, box, err)) return -1;
    } else {
      // input grid is (2*OH) x (2*OW); view it as [B, OH, 2, OW, (2, lda)] so that a stride-2 tap is a dense box
      const int IWin = 2 * d.OW, IHin = 2 * d.OH;
      const cuuint64_t dims[5] = {static_cast<cuuint64_t>(2) * d.lda, static_cast<cuuint64_t>(d.OW), 2,
                                  static_cast<cuuint64_t>(d.OH), static_cast<cuuint64_t>(d.B)};
      const cuuint64_t strides[4] = {static_cast<cuuint64_t>(2) * d.lda * 2, static_cast<cuuint64_t>(IWin) * d.lda * 2,
                                     static_cast<cuuint64_t>(2) * IWin * d.lda * 2,
                                     static_cast<cuuint64_t>(IHin) * IWin * d.lda * 2};
      const cuuint32_t box[5] = {BK, static_cast<cuuint32_t>(a.TW), 1, static_cast<cuuint32_t>(a.TH), 1};
      if (encode(&op->ta, d.dtype, 5, d.A, dims, strides, box, err)) return -1;
    }
  }

  const int bn = pick_bn(d.N, m_tiles);
  if (d.stats_out && d.N % bn != 0) { *err = "gemm: a LayerNorm-statistics producer needs N to be a multiple of its n-tile (equal-width partials)"; return -1; }
  op->bn = bn;
  a.n_tiles = (d.N + bn - 1) / bn;
  {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(d.K), static_cast<cuuint64_t>(d.N)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(d.K) * 2};
    const cuuint32_t box[2] = {BK, static_cast<cuuint32_t>(bn / 2)};      // each CTA of a pair loads half of the n-tile
    if (encode(&op->tb, d.dtype, 2, d.W, dims, strides, box, err)) return -1;
  }
  const int stage_bytes = A_STAGE_BYTES + (bn / 2) * BK * 2;
  const size_t vec_bytes = 3 * 4 * static_cast<size_t>(a.n_tiles) * bn;     // bias | gamma | colsum for all n-tiles
  int stages = static_cast<int>((206 * 1024 - vec_bytes) / stage_bytes);
  stages = std::min(stages, MAX_STAGES);
  stages = std::max(2, std::min(stages, std::max(2, 2 * a.kblocks)));
  a.stages = stages;
  a.m_tiles = m_tiles;
  op->smem = 1024 + static_cast<size_t>(stages) * stage_bytes + 256 + vec_bytes;
  const long long ptiles = static_cast<long long>((m_tiles + 1) / 2) * a.n_tiles;
  op->grid = 2u * static_cast<unsigned>(std::min<long long>(ptiles, num_sms() / 2));
  // epilogue groups on alternate tiles once a CTA pair has at least six tiles to walk (see the kernel); the LayerNorm
  // partials a producer writes per row follow: one per (n-tile, column half) or one per (n-tile, column half, group)
  a.epi_groups = ptiles >= 6LL * (op->grid / 2) ? 2 : 1;
  a.stats_parts_out = a.n_tiles * (a.epi_groups == 2 ? 2 : 4);
  op->flops = 2.0 * d.M * static_cast<double>(d.N) * d.K;
  return 0;
}

template <typename T, int BN, int EP>
static int launch_inst(const GemmOp& op, cudaStream_t st) {
  if (int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(gemm_tc_kernel<T, BN, EP>), 226 * 1024)) return e;
  launch_k(gemm_tc_kernel<T, BN, EP>, dim3(op.grid), dim3(GEMM_THREADS), op.smem, st, op.ta, op.tb, op.args);
  return static_cast<int>(cudaGetLastError());
}

static int pick_ep(const GemmArgs& a) {
  const bool special_rows = a.out_fp32 || a.remap_rows || a.shuffle_cout > 0 || a.hm_S > 0 || a.row_zero != nullptr;
  if (special_rows) return EP_GENERIC;
  if (a.stats_in) {
    if (a.gamma || a.resid || a.stats_out) return EP_GENERIC;
    if (a.act == ACT_NONE) return EP_LN;
    if (a.act == ACT_GELU) return EP_LN_GELU;
    return EP_GENERIC;
  }
  if (a.gamma || a.resid || a.stats_out) return a.act == ACT_NONE ? EP_RESID : EP_GENERIC;
  return a.act == ACT_NONE ? EP_BIAS : EP_BIAS_ACT;
}

template <typename T, int BN>
static int launch_ep(const GemmOp& op, cudaStream_t st) {
  switch (pick_ep(op.args)) {
    case EP_BIAS: return launch_inst<T, BN, EP_BIAS>(op, st);
    case EP_BIAS_ACT: return launch_inst<T, BN, EP_BIAS_ACT>(op, st);
    case EP_LN: return launch_inst<T, BN, EP_LN>(op, st);
    case EP_LN_GELU: return launch_inst<T, BN, EP_LN_GELU>(op, st);
    case EP_RESID: return launch_inst<T, BN, EP_RESID>(op, st);
    default: return launch_inst<T, BN, EP_GENERIC>(op, st);
  }
}

int gemm_launch(const GemmOp& op, cudaStream_t st) {
#define LWB_BN_SWITCH(T)                                     \
  switch (op.bn) {                                           \
    case 64: return launch_ep<T, 64>(op, st);                \
    case 128: return launch_ep<T, 128>(op, st);              \
    case 192: return launch_ep<T, 192>(op, st);              \
    case 256: return launch_ep<T, 256>(op, st);              \
    default: return -1;                                      \
  }
  if (op.dtype == DT_BF16) { LWB_BN_SWITCH(__nv_bfloat16) } else { LWB_BN_SWITCH(__half) }
#undef LWB_BN_SWITCH
}

}  // namespace lwb
