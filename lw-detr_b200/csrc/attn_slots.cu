// tcgen05 / TMA attention for head dims 16 and 32 - the ViT window attention (vit.py:130-137 with B' = 16B, N = 100) and
// the ViT global attention (vit.py:201-204) of LW-DETR-tiny / small / medium / large.  At these head dims the kernel is
// bound by the exponentials, not by the tensor core (16 MUFU.EX2 per clock and SM against <= 0.5 k clocks of MMA per
// 128x128 score tile), so the design is organised around the softmax threads (DESIGN.md 3.1, profiles/r02_attn_history.md):
//
//   * FOUR independent "slots" per CTA (one CTA per SM, 20 warps).  A slot owns one 128-row query tile, its own 128 TMEM
//     columns (S 64 fp32 | P 32 packed 16-bit | O dh fp32 | row sums 16) and its own barrier set; keys come in chunks of 64.
//   * warps 0-15 : SOFTMAX warps, four per slot (slot = warp / 4, TMEM lane quarter = warp % 4), ONE THREAD PER QUERY ROW
//                  (tcgen05.ld 32x32b hands thread t row t): the row maximum, the lazy rescale decision (FlashAttention-4:
//                  the reference maximum only moves when exceeded by 2^8) and P need no cross-thread exchange at all.
//                  Every scheduler hosts one softmax warp of each slot, i.e. four independent instruction streams.
//   * warps 16-19: one DRIVER thread per slot: its tcgen05.mma (S = Q K^T, O += P V with P read from TMEM), its TMA loads
//                  straight out of the packed [rows, 3C] qkv matrix (Q double-buffered one item ahead, K/V ring probed
//                  without blocking) and the commits.  This lone thread is the slot's critical path (one dependent
//                  instruction per 10-20 clocks): everything it does per chunk is incremental.
//   * row sums out of the P V product (head dim 16): the B operand is [V | 1] with N = 32, the block of ones reached through
//     the descriptor's leading byte offset.
//   * exp2: packed fp32x2 FMAs (fma.rn.f32x2) fold scale and max-subtraction, every exponential on the MUFU.
//   * setmaxnreg moves registers from the driver warps (96 -> 64) to the softmax warps (96 -> 104), which hold a 64-score row
//     chunk.  The pool is per CTA: what the 16 softmax warps take (16*32*8) must not exceed what the 4 driver warps release.
//
// Work decomposition: every slot walks its own (sequence, head, query tile) items with its own K/V ring.  LONG (template,
// chosen from the sequence length) = sequences of more than one tile (1600 tokens): warps whose rows lie beyond the sequence
// only keep the barrier protocol going; one-tile sequences (the 100-token windows) instead defer an item's epilogue into
// the next item's first chunk, and their tail chunk only exponentiates the valid keys (104 instead of 128).
// CTAs are persistent and walk their items with a fixed stride.
#include "attn.h"
#include "launch.h"
#include "ptx.cuh"
#include "tma_util.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

namespace lwb {
namespace sl {

static constexpr int SLOTS = 4;
static constexpr int BM = 128;                 // query rows per slot
static constexpr int BK = 64;                  // keys per chunk
static constexpr int W_DRIVER = 4 * SLOTS;      // warps 0-15: softmax (slot = warp / 4, TMEM lane quarter = warp % 4); 16-19: one driver per slot
static constexpr int THREADS = 32 * (W_DRIVER + SLOTS);
static constexpr float LAZY_LOG2 = 8.f;        // the row reference maximum moves only when exceeded by more than 2^8

template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

// Debug aid (LWDETR_B200_DEBUG_WAIT=1): barrier waits time out after ~50 ms and leave a record (source line, CTA, warp,
// parity) in MAPPED HOST memory before trapping - readable after the device fault, see attention_slots_debug_dump().
struct WaitDbg {
  unsigned int n;
  unsigned int rec[64][4];
};

// Barrier operations on precomputed 32-bit shared addresses: the generic-pointer forms re-derive the address (cvta, CTA-id
// mapping, alignment arithmetic) at every use when registers are tight - ncu counted ~115 of 400 instructions per chunk of a
// softmax thread in synchronisation code that should be a dozen.
__device__ __forceinline__ bool try_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool test_a(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must surface as a trap (CUDA error), never as a hung GPU.  The spin is try_wait + counter +
// branch (try_wait itself suspends the thread for a while); after 2^26 failed tries (>= 0.5 s) the thread traps, leaving a
// record (source line, CTA, thread, parity) in mapped host memory when the debug buffer exists.
__device__ __forceinline__ void wait_a(uint32_t bar, uint32_t parity, WaitDbg* dbg, int tag) {
  if (try_wait_a(bar, parity)) return;
  uint32_t spins = 0;
  while (!try_wait_a(bar, parity)) {
    if (++spins > (dbg != nullptr ? (1u << 21) : (1u << 26))) {
      if (dbg != nullptr) {
        const unsigned i = atomicAdd(&dbg->n, 1u);
        if (i < 64) {
          dbg->rec[i][0] = static_cast<unsigned>(tag);
          dbg->rec[i][1] = blockIdx.x;
          dbg->rec[i][2] = threadIdx.x;
          dbg->rec[i][3] = parity;
        }
        __threadfence_system();
      }
      __trap();
    }
  }
}
__device__ __forceinline__ void arrive_a(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void commit_a(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_2d_a(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

#define SL_WAIT(bar, par) wait_a(bar, par, p.dbg, __LINE__)

struct SlotArgs {
  WaitDbg* dbg;
  void* o;
  int ldo;
  int seqlen, nseq, heads;
  float scale_log2;
  int C;          // column distance between the q, k and v blocks of the packed matrix
  int qtiles;     // 128-row query tiles per sequence
  int nitems;     // nseq*heads*qtiles (slot items)
};

template <int DH>
struct Geo {
  static constexpr int STAGES = 4;
  static constexpr int NRINGS = SLOTS;
  static constexpr int Q_BYTES = BM * DH * 2;
  static constexpr int KV_BYTES = BK * DH * 2;                 // one K (or V) chunk
  static constexpr int STAGE_BYTES = 2 * KV_BYTES;
  static constexpr int SMEM_Q = SLOTS * 2 * Q_BYTES;
  static constexpr int SMEM_RING = NRINGS * STAGES * STAGE_BYTES;
  static constexpr int NBAR = 10 * SLOTS + 2 * NRINGS * STAGES;
  static constexpr int SMEM = 1024 + SMEM_Q + SMEM_RING + 1024 + 512 + 64;  // ... | barriers + TMEM slot (1 KB) | ones tile (512 B)
  static_assert(NBAR * 8 + 16 <= 1024, "barrier block");
  static constexpr uint32_t SLOT_COLS = 128;                   // S 64 | P 32 | O DH (<= 32): four slots fill the 512 columns
};

template <typename T, int DH, bool LONG>   // LONG: sequences of more than one 128-row tile
__global__ void __launch_bounds__(THREADS, 1) attn_slots_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                                                                const SlotArgs p) {
  using G = Geo<DH>;
  constexpr int STAGES = G::STAGES;
  constexpr uint32_t PITCH = DH * 2;
  constexpr uint32_t LAYOUT = DH == 64 ? 2u : (DH == 32 ? 4u : 6u);   // SWIZZLE_128B / 64B / 32B
  constexpr uint32_t SBO = 8 * PITCH;
  constexpr uint32_t COL_S = 0, COL_P = 64, COL_O = 96, COL_L = 112;
  // Head dim 16 leaves 16 TMEM columns per slot: the row sums l = sum_k P come from the tensor core too instead of one FADD2
  // per pair in the softmax threads, whose instruction stream is what bounds the kernel.  A 16 x 16 tile of ones is appended
  // to the V tile - the B operand of O += P V becomes [V | 1] with N = 32 (second MN atom = the ones block, reached through
  // the descriptor's leading byte offset), so the SAME four MMAs per chunk produce O in columns 96-111 and the row sums in
  // columns 112-127 (a tcgen05.mma costs the same ~45 clk for any N <= 64).  l is then the sum of the ROUNDED P, exactly
  // what the P V product sees.  At head dim 32 the columns are taken by O and the sums stay in registers.
  constexpr bool SUMS = DH == 16;
  extern __shared__ uint8_t sl_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(sl_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                                          // [slot][2][Q_BYTES]
  uint8_t* sRing = sQ + G::SMEM_Q;                             // [ring][stage][K | V]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRing + G::SMEM_RING);
  uint64_t* q_full = bars;                 // [slot][2 buffers]
  uint64_t* q_empty = q_full + 2 * SLOTS;  // [slot][2]: the item's last S MMA has read the Q tile
  uint64_t* s_full = q_empty + 2 * SLOTS;  // S(j) written by the tensor core
  uint64_t* s_free = s_full + SLOTS;       // the slot's four softmax warps hold S(j) in registers
  uint64_t* p_full = s_free + SLOTS;       // P(j) stored (and O rescaled if the reference maximum moved)
  uint64_t* p_empty = p_full + SLOTS;      // PV(j) completed: P may be overwritten, O is current
  uint64_t* o_full = p_empty + SLOTS;      // all PV of the item completed
  uint64_t* o_free = o_full + SLOTS;       // O read out: the next item may overwrite it
  uint64_t* kv_full = o_free + SLOTS;      // [ring][stage]
  uint64_t* kv_empty = kv_full + G::NRINGS * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(kv_empty + G::NRINGS * STAGES);
  uint8_t* sOnes = sRing + G::SMEM_RING + 1024;                  // 16 x 16 ones (512 B, 256-byte aligned), behind the 1 KB barrier block

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    for (int s = 0; s < SLOTS; ++s) {
      for (int b = 0; b < 2; ++b) {
        mbar_init(&q_full[s * 2 + b], 1);
        mbar_init(&q_empty[s * 2 + b], 1);
      }
      mbar_init(&s_full[s], 1);
      mbar_init(&s_free[s], 4);
      mbar_init(&p_full[s], 4);
      mbar_init(&p_empty[s], 1);
      mbar_init(&o_full[s], 1);
      mbar_init(&o_free[s], 4);
    }
    for (int i = 0; i < G::NRINGS * STAGES; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == W_DRIVER) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (SUMS && threadIdx.x < 128) {
    reinterpret_cast<uint32_t*>(sOnes)[threadIdx.x] = Cvt<T>::pack(1.f, 1.f);
    fence_proxy_async_smem();                                    // generic-proxy writes -> visible to the tensor core's reads
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_sync();   // the prologue above touched no global data; everything below reads the predecessor's output
  // 32-bit shared addresses of the barrier arrays (8 bytes per barrier)
  const uint32_t a_bars = smem_u32(bars);
  const uint32_t a_q_full = a_bars, a_q_empty = a_q_full + 16 * SLOTS, a_s_full = a_q_empty + 16 * SLOTS, a_s_free = a_s_full + 8 * SLOTS;
  const uint32_t a_p_full = a_s_free + 8 * SLOTS, a_p_empty = a_p_full + 8 * SLOTS, a_o_full = a_p_empty + 8 * SLOTS, a_o_free = a_o_full + 8 * SLOTS;
  const uint32_t a_kv_full = a_o_free + 8 * SLOTS, a_kv_empty = a_kv_full + 8 * G::NRINGS * STAGES;

  const int nchunks = (p.seqlen + BK - 1) / BK;
  struct ItemIt {
    int seq, head, qtile;
  };
  // item -> (sequence, head, query tile)
  auto decode = [&](int item, ItemIt& it) {
    it.qtile = item % p.qtiles;
    const int sh = item / p.qtiles;
    it.head = sh % p.heads;
    it.seq = sh / p.heads;
  };
  // Walking items first, first + stride, ... without a division per item (three divisions per item in every softmax thread
  // and driver cursor were a measurable share of the 2-chunk window items): the stride is decomposed once into (sequences,
  // heads, query tiles) and added with carries.
  const int stride = static_cast<int>(gridDim.x) * SLOTS;
  const int per_seq = p.heads * p.qtiles;
  const int st_seq = stride / per_seq;
  const int st_rem = stride - st_seq * per_seq;
  const int st_head = st_rem / p.qtiles;
  const int st_qt = st_rem - st_head * p.qtiles;
  auto it_advance = [&](ItemIt& it) {
    it.qtile += st_qt;
    if (it.qtile >= p.qtiles) {
      it.qtile -= p.qtiles;
      ++it.head;
    }
    it.head += st_head;
    if (it.head >= p.heads) {
      it.head -= p.heads;
      ++it.seq;
    }
    it.seq += st_seq;
  };
  // items of slot sl: first, first + stride, ...
  auto first_of = [&](int sl) { return static_cast<int>(blockIdx.x) * SLOTS + sl; };
  auto count_of = [&](int sl) { const int f = first_of(sl); return f < p.nitems ? (p.nitems - f + stride - 1) / stride : 0; };

  if (warp >= W_DRIVER) {
    reg_dec<64>();
    if (lane == 0) {
      // ---------------------------------------------------------------- driver of one slot: its tcgen05.mma, its TMA loads.
      // The slot's work is a flat stream of (item, chunk) steps; S is issued one chunk ahead of the softmax warps, P V follows
      // them, loads run ahead as far as the ring allows (non-blocking probe).  This thread's own instruction stream is the
      // critical path of the slot - ncu of the first version (profiles/r02_attn_history.md) showed the softmax warps
      // waiting for S a quarter of their time while the lone driver thread worked through ~250 instructions per chunk at
      // one dependent instruction per 10-20 clocks - so everything per chunk is incremental: no divisions, no descriptor
      // rebuilds, stage / phase counters that wrap by comparison.
      const int slot = warp - W_DRIVER;
      const uint32_t tslot = tmem + static_cast<uint32_t>(slot) * G::SLOT_COLS;
      constexpr bool BF = Cvt<T>::is_bf16;
      constexpr uint32_t idesc_s = umma_idesc_f16(BF, BM, BK);                 // S: N = 64 keys, Q and K both K-major
      constexpr uint32_t idesc_o = umma_idesc_f16(BF, BM, SUMS ? 32 : DH) | (1u << 16);    // O: B (= V, or [V | ones]) is MN-major
      uint8_t* ring = sRing + slot * STAGES * G::STAGE_BYTES;
      const uint32_t a_ring = smem_u32(ring), a_q = smem_u32(sQ + slot * 2 * G::Q_BYTES);
      const uint32_t rfull = a_kv_full + 8 * slot * STAGES, rempty = a_kv_empty + 8 * slot * STAGES;
      const uint32_t b_q_full = a_q_full + 16 * slot, b_q_empty = a_q_empty + 16 * slot;
      const uint32_t b_s_full = a_s_full + 8 * slot, b_s_free = a_s_free + 8 * slot, b_p_full = a_p_full + 8 * slot, b_p_empty = a_p_empty + 8 * slot;
      const uint32_t b_o_full = a_o_full + 8 * slot, b_o_free = a_o_free + 8 * slot;
      const int first = first_of(slot);
      const int n_my = count_of(slot);
      const uint32_t total = static_cast<uint32_t>(n_my) * nchunks;
      // descriptors of stage 0; a stage further on adds STAGE_BYTES to the start address (and, with the row sums, takes the
      // same amount off the leading byte offset that reaches the fixed block of ones)
      constexpr uint64_t STAGE_D = G::STAGE_BYTES >> 4;
      const uint64_t qd[2] = {umma_desc(a_q, SBO, LAYOUT), umma_desc(a_q + G::Q_BYTES, SBO, LAYOUT)};
      const uint64_t kd0 = umma_desc(a_ring, SBO, LAYOUT);
      const uint32_t vaddr0 = a_ring + G::KV_BYTES;
      uint64_t vd0[BK / 16];
#pragma unroll
      for (int kk = 0; kk < BK / 16; ++kk) {
        const uint32_t va = vaddr0 + 16 * PITCH * kk;
        vd0[kk] = SUMS ? umma_desc_lbo(va, SBO, LAYOUT, smem_u32(sOnes) - va) : umma_desc(va, SBO, LAYOUT);
      }
      constexpr uint64_t V_STEP = SUMS ? (STAGE_D - (STAGE_D << 16)) : STAGE_D;

      // ---- loads.  K/V: fill f of the ring goes to stage f mod STAGES in round f / STAGES
      uint32_t l_f = 0, l_st = 0, l_ph = 0;
      int l_i = 0, l_j = 0, l_row = 0, l_col = 0;
      ItemIt l_it{0, 0, 0}, q_it{0, 0, 0};
      if (n_my > 0) {
        decode(first, l_it);
        q_it = l_it;
      }
      auto l_seek = [&]() {                                          // normalise (l_i, l_j) and look up the item's K/V rows
        while (l_j >= nchunks) {
          l_j -= nchunks;
          ++l_i;
          it_advance(l_it);
        }
        if (l_i < n_my) {
          l_row = l_it.seq * p.seqlen;
          l_col = l_it.head * DH;
        }
      };
      l_seek();
      auto top_up = [&]() {
        while (l_i < n_my) {
          if (l_f >= static_cast<uint32_t>(STAGES) && !test_a(rempty + 8 * l_st, l_ph ^ 1u)) break;
          const uint32_t dst = a_ring + l_st * G::STAGE_BYTES;
          const int row = l_row + l_j * BK;
          expect_tx_a(rfull + 8 * l_st, G::STAGE_BYTES);
          tma_2d_a(dst, &tmKV, rfull + 8 * l_st, p.C + l_col, row);
          tma_2d_a(dst + G::KV_BYTES, &tmKV, rfull + 8 * l_st, 2 * p.C + l_col, row);
          ++l_f;
          ++l_st;
          if (l_st >= static_cast<uint32_t>(STAGES)) {
            l_st -= STAGES;
            l_ph ^= 1u;
          }
          ++l_j;
          if (l_j >= nchunks) l_seek();
        }
      };
      // Q: two buffers, requested one item ahead
      uint32_t aq = 0;                 // Q tiles requested
      int q_i = 0;                     // next item whose Q tile is to be requested
      auto load_next_q = [&]() {
        if (q_i >= n_my) return;
        const uint32_t buf = aq & 1;
        if (aq >= 2) SL_WAIT(b_q_empty + 8 * buf, ((aq >> 1) - 1) & 1);
        expect_tx_a(b_q_full + 8 * buf, G::Q_BYTES);
        tma_2d_a(a_q + buf * G::Q_BYTES, &tmQ, b_q_full + 8 * buf, q_it.head * DH, q_it.seq * p.seqlen + q_it.qtile * BM);
        ++aq;
        ++q_i;
        it_advance(q_it);
      };

      int sj = 0, pj = 0;
      uint32_t s_st = 0, s_ph = 0, p_st = 0;
      uint32_t sc = 0, pc = 0;         // S / PV issued by this slot
      uint32_t as_item = 0;            // items whose S phase has completed
      uint32_t n_item = 0;             // items completed (o_full committed)
      auto issue_s = [&]() {           // S(sc) = Q K^T
        // The fill this S needs may be one this very thread still owes (its stage was not free at the last probe): keep
        // probing the ring while waiting - a blocking wait here could wait for itself.
        while (!try_wait_a(rfull + 8 * s_st, s_ph)) top_up();
        const uint32_t buf = as_item & 1;
        if (sj == 0) SL_WAIT(b_q_full + 8 * buf, (as_item >> 1) & 1);
        if (sc > 0) SL_WAIT(b_s_free, (sc - 1) & 1);                 // the softmax warps pulled the previous S out of TMEM
        tc_fence_after();
        const uint64_t kdesc = kd0 + STAGE_D * s_st;
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) umma_f16_ss(tslot + COL_S, qd[buf] + 2 * kk, kdesc + 2 * kk, idesc_s, kk != 0 ? 1u : 0u);
        commit_a(b_s_full);
        if (sj + 1 == nchunks) {                                     // last S of the item: its Q buffer may be refilled once these MMAs are done
          commit_a(b_q_empty + 8 * buf);
          ++as_item;
        }
        ++sc;
        if (++s_st == static_cast<uint32_t>(STAGES)) {
          s_st = 0;
          s_ph ^= 1u;
        }
        if (++sj == nchunks) sj = 0;
      };
      load_next_q();
      load_next_q();
      top_up();
      if (total > 0) issue_s();
      while (pc < total) {
        top_up();
        if (sc < total) issue_s();                                   // S(pc + 1) runs while the softmax warps work on S(pc)
        SL_WAIT(b_p_full, pc & 1);                                   // P(pc) is in TMEM, O carries the current reference maximum
        if (pj == 0 && n_item > 0) SL_WAIT(b_o_free, (n_item - 1) & 1);   // the previous item's O has been read out
        tc_fence_after();
        const uint32_t acc0 = pj != 0 ? 1u : 0u;
#pragma unroll
        for (int kk = 0; kk < BK / 16; ++kk)                         // 16 keys per MMA: A advances 8 TMEM columns, B 16 rows
          umma_f16_ts(tslot + COL_O, tslot + COL_P + 8 * kk, vd0[kk] + V_STEP * p_st, idesc_o, kk != 0 ? 1u : acc0);
        commit_a(b_p_empty);
        commit_a(rempty + 8 * p_st);
        if (pj + 1 == nchunks) {
          commit_a(b_o_full);
          ++n_item;
          load_next_q();                                             // the Q buffer of the item before this one is free by now
        }
        ++pc;
        if (++p_st == static_cast<uint32_t>(STAGES)) p_st = 0;
        if (++pj == nchunks) pj = 0;
      }
    }
  } else {
    reg_inc<104>();
    const int slot = warp >> 2;
    const uint32_t tslot = tmem + static_cast<uint32_t>(slot) * G::SLOT_COLS;
    const int first = first_of(slot);
    // ---------------------------------------------------------------------- softmax / epilogue: one thread per query row
    const int quarter = warp & 3;                                  // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;
    const uint32_t tbase = tslot + (static_cast<uint32_t>(quarter * 32) << 16);
    const float c = p.scale_log2;
    const uint64_t c2 = f2_pack(c, c);
    const uint32_t b_s_full = a_s_full + 8 * slot, b_s_free = a_s_free + 8 * slot, b_p_full = a_p_full + 8 * slot, b_p_empty = a_p_empty + 8 * slot;
    const uint32_t b_o_full = a_o_full + 8 * slot, b_o_free = a_o_free + 8 * slot;
    const bool elected = lane == 0;
    uint32_t n_c = 0, n_item = 0;
    ItemIt s_it{0, 0, 0};
    if (first < p.nitems) decode(first, s_it);
    // The epilogue of an item (wait for its last P V, read O and the row sum, store) is DEFERRED into the first chunk of the
    // slot's next item, between that chunk's exponentials and its P store: the P V round trip (driver wake-up + 4 MMAs +
    // commit, ~600 clk; 10 % of all samples of the 2-chunk window items sat in that wait) then hides behind exponentials.
    // Measured (isolated, L2 flushed): windows 51.2 -> 49.2 us (small), 112 -> 98 us (medium), 63.5 -> 57.4 us (large); the
    // long sequences lose 5 % to the extra live registers, so they keep the immediate epilogue (LONG).
    bool pend = false, pend_store = false;
    T* pend_dst = nullptr;
    uint64_t pend_lsum2 = 0;
    auto finish_item = [&]() {                                     // O / l -> global for the pending item
      SL_WAIT(b_o_full, n_item & 1);
      tc_fence_after();
      float inv;
      if (SUMS) {
        float l8[8];
        __syncwarp();
        tmem_ld_x8(tbase + COL_L, l8);                              // 16 identical columns: the row sum of the rounded P
        tmem_ld_wait();
        inv = 1.f / l8[0];
      } else {
        float l0, l1;
        f2_unpack(pend_lsum2, l0, l1);
        inv = 1.f / (l0 + l1);
      }
      U8 ov[DH / 16];
#pragma unroll
      for (int cc = 0; cc < DH / 16; ++cc) {
        float o16[16];
        __syncwarp();
        tmem_ld_x16(tbase + COL_O + cc * 16, o16);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i) ov[cc].v[i] = Cvt<T>::pack(o16[2 * i] * inv, o16[2 * i + 1] * inv);
      }
      tc_fence_before();
      __syncwarp();
      if (elected) arrive_a(b_o_free);
      ++n_item;
      if (pend_store) {
#pragma unroll
        for (int cc = 0; cc < DH / 16; ++cc) stg256(pend_dst + cc * 16, ov[cc]);
      }
      pend = false;
    };
    for (int item = first; item < p.nitems; item += stride) {
      const int seq = s_it.seq, head = s_it.head, qtile = s_it.qtile;
      it_advance(s_it);
      // A warp whose 32 rows all lie beyond the sequence (the second half of the last 128-row tile of a 1600-token sequence:
      // 2 of 52 warp-tiles) only keeps the barrier protocol going: no TMEM traffic, no exponentials, nothing stored.
      if (LONG && qtile * BM + quarter * 32 >= p.seqlen) {
        if (pend) finish_item();
        for (int j = 0; j < nchunks; ++j, ++n_c) {
          SL_WAIT(b_s_full, n_c & 1);
          if (elected) arrive_a(b_s_free);
          if (n_c > 0) SL_WAIT(b_p_empty, (n_c - 1) & 1);
          if (elected) arrive_a(b_p_full);
        }
        SL_WAIT(b_o_full, n_item & 1);
        if (elected) arrive_a(b_o_free);
        ++n_item;
        continue;
      }
      float m_ref = -INFINITY;
      uint64_t lsum2 = f2_pack(0.f, 0.f);
      for (int j = 0; j < nchunks; ++j, ++n_c) {
        float v[64];
        SL_WAIT(b_s_full, n_c & 1);
        tc_fence_after();
        tmem_ld_x32(tbase + COL_S, v);
        tmem_ld_x32(tbase + COL_S + 32, v + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (elected) arrive_a(b_s_free);                           // one elected arrival per warp
        const int nvalid = min(BK, p.seqlen - j * BK);             // keys >= nvalid belong to the next sequence / are padding
        // ---- row maximum of the valid keys.  Ragged chunks are handled in groups of 8 keys with warp-uniform branches:
        // full groups take the unmasked code, only the group that holds the boundary pays for per-key predicates.
        float mchunk;
        if (nvalid == BK) {
          float mm[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
          for (int i = 0; i < 16; i += 2)
#pragma unroll
            for (int q = 0; q < 4; ++q) mm[q] = fmaxf(mm[q], fmaxf(v[q * 16 + i], v[q * 16 + i + 1]));
          mchunk = fmaxf(fmaxf(mm[0], mm[1]), fmaxf(mm[2], mm[3]));
        } else {
          mchunk = -INFINITY;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            if (g * 8 + 8 <= nvalid) {
              mchunk = fmaxf(mchunk, fmaxf(fmaxf(fmaxf(v[g * 8], v[g * 8 + 1]), fmaxf(v[g * 8 + 2], v[g * 8 + 3])),
                                           fmaxf(fmaxf(v[g * 8 + 4], v[g * 8 + 5]), fmaxf(v[g * 8 + 6], v[g * 8 + 7]))));
            } else if (g * 8 < nvalid) {
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (g * 8 + e < nvalid) mchunk = fmaxf(mchunk, v[g * 8 + e]);
            }
          }
        }
        // lazy reference maximum: a row's decision only involves its own thread
        const bool move = (mchunk - m_ref) * c > LAZY_LOG2;        // true at j = 0 (m_ref = -inf)
        const float alpha = move ? ex2((m_ref - mchunk) * c) : 1.f;
        if (move) m_ref = mchunk;
        const float msc = m_ref * c;
        if (!SUMS && move) lsum2 = f2_fma(lsum2, f2_pack(alpha, alpha), f2_pack(0.f, 0.f));
        const uint64_t nm2 = f2_pack(-msc, -msc);
        uint32_t pk[32];
        auto group = [&](int g, auto masked_tag) {                 // keys 8g .. 8g+7 -> pk[4g .. 4g+3]
          constexpr bool MASKED = decltype(masked_tag)::value;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = g * 4 + q;                               // pair index: keys 2i, 2i+1
            float a0, a1;
            f2_unpack(f2_fma(f2_pack(v[2 * i], v[2 * i + 1]), c2, nm2), a0, a1);
            float e0 = ex2(a0), e1 = ex2(a1);
            if (MASKED) {
              e0 = 2 * i < nvalid ? e0 : 0.f;
              e1 = 2 * i + 1 < nvalid ? e1 : 0.f;
            }
            pk[i] = Cvt<T>::pack(e0, e1);
            if (!SUMS) lsum2 = f2_add(lsum2, f2_pack(e0, e1));
          }
        };
        if (nvalid == BK) {
#pragma unroll
          for (int g = 0; g < 8; ++g) group(g, std::false_type{});
        } else {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            if (g * 8 + 8 <= nvalid) {
              group(g, std::false_type{});
            } else if (g * 8 < nvalid) {
              group(g, std::true_type{});
            } else {
#pragma unroll
              for (int q = 0; q < 4; ++q) pk[g * 4 + q] = 0u;
            }
          }
        }
        // only now wait for PV(j-1): its latency hides behind the exponentials above (P is single-buffered)
        if (n_c > 0) SL_WAIT(b_p_empty, (n_c - 1) & 1);
        tc_fence_after();
        if (!LONG && j == 0 && pend) finish_item();                 // the previous item's last P V is complete at this point
        if (j > 0 && __any_sync(0xffffffffu, move)) {               // rare after the first chunks: rescale this row of O (and of l)
#pragma unroll
          for (int cc = 0; cc < (DH + (SUMS ? 16 : 0)) / 16; ++cc) {
            float o16[16];
            uint32_t u16[16];
            __syncwarp();
            tmem_ld_x16(tbase + COL_O + cc * 16, o16);              // COL_L directly follows O at head dim 16
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) u16[i] = __float_as_uint(o16[i] * alpha);
            tmem_st_x16(tbase + COL_O + cc * 16, u16);
          }
        }
        tmem_st_x16(tbase + COL_P, pk);
        tmem_st_x16(tbase + COL_P + 16, pk + 16);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (elected) arrive_a(b_p_full);
      }
      // ---- the item's epilogue is deferred (see finish_item above)
      const int qrow = qtile * BM + r;
      pend_dst = reinterpret_cast<T*>(p.o) + (static_cast<long long>(seq) * p.seqlen + qrow) * p.ldo + head * DH;
      pend_store = qrow < p.seqlen;
      pend_lsum2 = lsum2;
      pend = true;
      if (LONG) finish_item();        // 13+ chunks per item amortise the round trip; deferring only costs registers there (measured)
    }
    if (pend) finish_item();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_DRIVER) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

static WaitDbg* g_dbg_host = nullptr;
static WaitDbg* debug_buffer() {
  static WaitDbg* dev = [] () -> WaitDbg* {
    const char* e = getenv("LWDETR_B200_DEBUG_WAIT");
    if (!e || atoi(e) == 0) return nullptr;
    void* h = nullptr;
    void* d = nullptr;
    if (cudaHostAlloc(&h, sizeof(WaitDbg), cudaHostAllocMapped) != cudaSuccess) return nullptr;
    memset(h, 0, sizeof(WaitDbg));
    if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) return nullptr;
    g_dbg_host = static_cast<WaitDbg*>(h);
    return static_cast<WaitDbg*>(d);
  }();
  return dev;
}

template <typename T, int DH, bool LONG>
static int launch_m(const AttnArgs& a, int C, cudaStream_t st) {
  using G = Geo<DH>;
  CUtensorMap tq, tkv;
  std::string err;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(a.ldq), static_cast<cuuint64_t>(a.nseq) * a.seqlen};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(a.ldq) * 2};
  const cuuint32_t boxq[2] = {DH, BM}, boxkv[2] = {DH, BK};
  const int dt = Cvt<T>::is_bf16 ? DT_BF16 : DT_F16;
  if (tma_encode(&tq, dt, 2, a.q, dims, strides, boxq, DH * 2, &err)) return -3;
  if (tma_encode(&tkv, dt, 2, a.q, dims, strides, boxkv, DH * 2, &err)) return -3;
  SlotArgs p;
  p.dbg = debug_buffer();
  p.o = a.o; p.ldo = a.ldo; p.seqlen = a.seqlen; p.nseq = a.nseq; p.heads = a.heads; p.scale_log2 = a.scale_log2; p.C = C;
  p.qtiles = (a.seqlen + BM - 1) / BM;
  const long long nitems = static_cast<long long>(a.nseq) * a.heads * p.qtiles;
  if (nitems > 0x7fffffffLL / 2) return -2;
  p.nitems = static_cast<int>(nitems);
  // One CTA per SM (it allocates all 512 TMEM columns): more than half of the shared memory is requested so that a second
  // CTA can never become resident and spin inside tcgen05.alloc.
  const size_t smem = std::max<size_t>(G::SMEM, 116 * 1024);
  if (int e = ensure_max_dyn_smem(reinterpret_cast<const void*>(attn_slots_kernel<T, DH, LONG>), 227 * 1024)) return e;
  const long long ctas = (nitems + SLOTS - 1) / SLOTS;
  const unsigned grid = static_cast<unsigned>(std::min<long long>(ctas, current_device_sms()));
  launch_k(attn_slots_kernel<T, DH, LONG>, dim3(grid), dim3(THREADS), smem, st, tq, tkv, p);
  return static_cast<int>(cudaGetLastError());
}

template <typename T, int DH>
static int launch(const AttnArgs& a, int C, cudaStream_t st) {
  return a.seqlen > BM ? launch_m<T, DH, true>(a, C, st) : launch_m<T, DH, false>(a, C, st);
}

}  // namespace sl

// prints (stderr) the barrier waits that timed out under LWDETR_B200_DEBUG_WAIT=1; returns their number
int attention_slots_debug_dump() {
  if (!sl::g_dbg_host) return 0;
  const unsigned n = sl::g_dbg_host->n;
  for (unsigned i = 0; i < n && i < 64; ++i)
    fprintf(stderr, "attn_slots wait timeout: line %u  cta %u  thread %u (warp %u)  parity %u\n", sl::g_dbg_host->rec[i][0], sl::g_dbg_host->rec[i][1],
            sl::g_dbg_host->rec[i][2], sl::g_dbg_host->rec[i][2] >> 5, sl::g_dbg_host->rec[i][3]);
  return static_cast<int>(n);
}

// Packed-qkv path for head dims 16 / 32: q, k, v are the column blocks [0,C), [C,2C), [2C,3C) of one 16-bit matrix.
int attention_slots_launch(int dtype, const AttnArgs& a, int dh, int C, cudaStream_t st) {
  if (dtype == DT_BF16) {
    if (dh == 16) return sl::launch<__nv_bfloat16, 16>(a, C, st);
    if (dh == 32) return sl::launch<__nv_bfloat16, 32>(a, C, st);
  } else {
    if (dh == 16) return sl::launch<__half, 16>(a, C, st);
    if (dh == 32) return sl::launch<__half, 32>(a, C, st);
  }
  return -2;
}

}  // namespace lwb
