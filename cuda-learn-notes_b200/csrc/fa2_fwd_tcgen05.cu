// FlashAttention-2 forward for B200 (sm_100a):  O = softmax(Q K^T * scale) V,  [B,H,N,D] fp16, non-causal.
//
// One CTA owns 256 query rows of one (batch, head): two 128-row Q tiles that share every K/V tile.
//   warp 0        TMA producer: Q tiles once, then rings of K and V tiles (BC keys each), 128B/64B-swizzled smem
//   warp 1        MMA issuer (one thread):  S_i = Q_i K_j^T   (tcgen05.mma SS, fp32 accumulate, 128 x BC into TMEM)
//                                            O_i += P_ij V_j   (tcgen05.mma TS: P read from TMEM, V MN-major smem)
//   warp 2        TMEM allocator
//   warp 3        masked build with seqlens_k only: zeroes the V rows past the length in the last KV tile
//   warps 4..7    softmax warpgroup for Q tile 0, one thread per query row: tcgen05.ld the S row, online softmax
//   warps 8..11   softmax warpgroup for Q tile 1       (row max / exp2 / row sum in fp32 registers), P written as
//                 fp16 into its OWN TMEM columns with tcgen05.st; O is rescaled in TMEM only when the row max grew
//                 by more than 2^8 (lazy rescaling); the same threads normalise and store O at the end (TMA store).
// TMEM columns (512 per SM), BC = 128 keys per KV tile except D = 96 (BC = 64):
//   D <= 96:  S0 S1 (2 x BC fp32) | P0 P1 (2 x BC/2, packed fp16) | O0 O1 (2 x D fp32).  P does not alias S, so the
//             scores of KV tile j+1 are produced while the softmax warps still work on tile j: the S columns are
//             handed back right after the row has been read into registers (s_free).
//   D = 128:  S (ONE buffer, BC fp32) | P0 P1 | O0 O1 = 128 + 128 + 256.  The two Q tiles take turns on the S buffer:
//             S_1(j) is issued once tile 0's warps hold S_0(j) in registers, S_0(j+1) once tile 1's hold S_1(j).
//             The next scores of a tile therefore never wait for its own PV (as they must when P aliases S), and
//             the two tiles run half a period apart, so their exponentials rarely compete for the MUFU pipe.
//             (+12 % over the S0 S1 O0 O1 / P-aliases-S layout, which is kept as variant 0x400.)
// P is handed to the MMA thread in pieces (two per KV tile for D <= 96: PV of the first half runs under the
// exponentials of the second; one for D = 128, where PV is off the critical chain).
//
// Replaces kernels/flash-attn/mma/basic/flash_attn_mma_share_qkv.cu:L45-709 (kernel) / L711-886 (launcher) and the
// other flash_attn_mma_stages_* variants (same math, different Ampere smem strategies).  Numerics follow the
// reference where it matters: scores scaled by 1/sqrt(D), softmax statistics in fp32, P rounded to fp16 before PV
// (share_qkv.cu:L431-478); the MMA accumulators are fp32 here (the reference default is fp16 accumulate).
#include <cmath>
#include <mutex>
#include <set>
#include <utility>

#include "abi_common.cuh"
#include "ptx.cuh"

namespace b200k {

template <int D_, int BC_, int STAGES_, bool V_DN_ = false, bool ALIAS_P_ = false, bool SHARE_S_ = false, int DT_ = 0>
struct Fa2Cfg {
  static constexpr int D = D_;
  static constexpr int DT = DT_;  // 0: fp16 Q/K/V/O and P; 1: bf16 (same kernel: kind::f16 with bf16 operand formats)
  static constexpr int BC = BC_;                       // keys per KV tile
  static constexpr int STAGES = STAGES_;
  // ALIAS_P: P overwrites the first BC/2 columns of S (needed when S0 S1 O0 O1 already fill the 512 columns, i.e.
  // D = 128 with BC = 128).  S_i(j+1) can then only be issued after PV_i(j), as in-order tcgen05 execution protects P.
  static constexpr bool ALIAS_P = ALIAS_P_;
  // SHARE_S: ONE S buffer used by both Q tiles in turn (S | P0 P1 | O0 O1 = BC + BC + 2 D columns: the other way to fit
  // D = 128 with BC = 128).  S_0(j+1) only needs the buffer back from tile 1 (its warps have S_1(j) in registers) and
  // NOT PV_0(j), so the chain  S -> softmax -> PV -> next S  of ALIAS_P is cut: the next scores are computed while the
  // softmax of the current ones runs.  The two tiles then necessarily run half a period apart (ping-pong), which
  // also keeps their exponentials from competing for the MUFU pipe.
  static constexpr bool SHARE_S = SHARE_S_;
  static_assert(!(ALIAS_P && SHARE_S), "pick one");
  static constexpr bool V_DN = V_DN_;  // V passed transposed as [B,H,D,N] (the reference's *_swizzle_qkv entry points)
  static constexpr int CW = (D % 64 == 0) ? 64 : 32;  // width of one smem chunk along D (elements)
  static constexpr int NCH = D / CW;
  static constexpr int ROWB = CW * 2;                  // bytes per smem row = swizzle span (128 or 64)
  static constexpr uint32_t SWZ_MODE = (ROWB == 128) ? 2u : 4u;
  static constexpr int BR = 128;                       // query rows per tile (= TMEM lanes)
  static constexpr int Q_CHUNK_BYTES = 128 * ROWB;     // one TMA box of Q: 128 rows x CW elements
  static constexpr int Q_TILE_BYTES = NCH * Q_CHUNK_BYTES;
  static constexpr int KV_CHUNK_BYTES = BC * ROWB;     // one TMA box of K or V: BC rows x CW elements
  static constexpr int KV_TILE_BYTES = NCH * KV_CHUNK_BYTES;  // = BC * D * 2 (also for the transposed-V layout)
  static constexpr int BAR_BYTES = 1024;
  static constexpr int SMEM_BYTES = 1024 + BAR_BYTES + 2 * Q_TILE_BYTES + 2 * STAGES * KV_TILE_BYTES;
  static constexpr int NS = SHARE_S ? 1 : 2;           // S buffers
  static constexpr int S_COL0 = 0, S_COL1 = SHARE_S ? 0 : BC;
  static constexpr int P_COL0 = ALIAS_P ? S_COL0 : NS * BC, P_COL1 = ALIAS_P ? S_COL1 : NS * BC + BC / 2;
  static constexpr int O_COL0 = ALIAS_P ? 2 * BC : (NS + 1) * BC, O_COL1 = O_COL0 + D;
  static constexpr int TMEM_COLS = 512;
  static constexpr int THREADS = 384;
  static_assert(D % 32 == 0 && D >= 32 && D <= 128, "head dim");
  static_assert(BC == 64 || BC == 128, "keys per tile");
  static_assert((ALIAS_P ? 2 : NS + 1) * BC + 2 * D <= 512, "TMEM columns");
  static_assert(SMEM_BYTES <= 232448, "smem");
};

// Lazy-rescale threshold in log2 units: P may grow up to 2^8 before the running max is moved (fp16 P and fp32 sums
// have ample range), so the O accumulator is touched only on the first few KV tiles of a row.
constexpr float kRescaleThreshold = 8.0f;

// Optional cycle trace of CTA (0,0) for pipeline analysis (tools/gpu_trace_fa2.py): trace[role][j][event] = clock64(),
// role 0 = MMA thread, 1 = softmax warp 4 (Q tile 0), 2 = softmax warp 8 (Q tile 1); first kTraceIters KV tiles.
constexpr int kTraceIters = 32, kTraceEvents = 8;
static unsigned long long* g_fa2_trace = nullptr;  // set through b200k_debug_set_trace()

// Masks (SURVEY 8f-4; the reference has none).  causal: query row r attends keys <= r; KV tiles entirely above the
// diagonal of BOTH Q tiles of the CTA are never loaded or multiplied (half the work at large N), tiles that touch the
// diagonal get an element mask.  seqlens (int32 [B], optional): keys >= seqlens[b] are masked for batch b ("varlen" in
// the padded [B,H,N,D] layout, i.e. a key-padding mask); every query row of the batch is still computed.
struct Fa2Mask {
  const int* seqlens = nullptr;
  int H = 1;
  int causal = 0;
};

// Zeroes keys [valid, BC) of the V tile at shared address vt, by the 32 lanes t of one warp, and makes the zeros visible
// to the tensor core (the caller's next mbarrier arrive orders them before the MMA).
template <class Cfg>
__device__ __forceinline__ void fa2_zero_v_keys(uint32_t vt, int valid, int t) {
  constexpr int D = Cfg::D, BC = Cfg::BC, ROWB = Cfg::ROWB;
  if constexpr (Cfg::V_DN) {
    // [D rows x 64 keys] boxes, 128B swizzle: the 8-key piece g of row d sits in 16-byte slot (g % 8) ^ (d % 8)
    for (int u = (valid / 8) * D + t; u < (BC / 8) * D; u += 32) {
      const int g = u / D, d = u % D, key0 = g * 8;
      const uint32_t addr = vt + (g / 8) * (D * 128) + d * 128 + (((g % 8) ^ (d % 8)) << 4);
      if (key0 >= valid) {
        st_shared_v4(addr, 0u, 0u, 0u, 0u);
      } else {
        for (int e = valid - key0; e < 8; ++e) st_shared_u16(addr + 2 * e, 0);
      }
    }
  } else {
    // a key is one ROWB-byte row of every CW-wide chunk; the swizzle only permutes 16-byte pieces inside a row
    for (int u = valid * (ROWB / 16) + t; u < BC * (ROWB / 16); u += 32)
#pragma unroll
      for (int c = 0; c < Cfg::NCH; ++c) st_shared_v4(vt + c * Cfg::KV_CHUNK_BYTES + u * 16, 0u, 0u, 0u, 0u);
  }
  fence_proxy_async_smem();
}

template <class Cfg, bool TRACE, int POLY, int NP, bool MASKED = false>
__global__ void __launch_bounds__(Cfg::THREADS, 1)
fa2_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                       const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, int N,
                       float scale_log2, unsigned long long* trace, const Fa2Mask mask) {
  auto tr = [&](int role, int j, int ev) {
    if constexpr (TRACE) {
      if (blockIdx.x == 0 && blockIdx.y == 0 && j < kTraceIters)
        trace[(role * kTraceIters + j) * kTraceEvents + ev] = clock64();
    }
  };
  constexpr int D = Cfg::D, BC = Cfg::BC, STAGES = Cfg::STAGES, NCH = Cfg::NCH, CW = Cfg::CW, ROWB = Cfg::ROWB;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw_addr);

  // barriers (8 bytes each)
  const uint32_t bar_q_full = base;                       // 2
  const uint32_t bar_k_full = base + 16;                  // STAGES
  const uint32_t bar_k_empty = bar_k_full + 8 * STAGES;   // STAGES
  const uint32_t bar_v_full = bar_k_empty + 8 * STAGES;   // STAGES
  const uint32_t bar_v_empty = bar_v_full + 8 * STAGES;   // STAGES
  const uint32_t bar_s_full = bar_v_empty + 8 * STAGES;   // 2   S_i(j) ready                 (MMA -> softmax i)
  const uint32_t bar_s_free = bar_s_full + 32;            // 2   S_i(j) is in registers       (softmax i -> MMA)
  const uint32_t bar_p_full = bar_s_free + 32;            // 2x4 piece p of P_i(j) written (and O_i rescaled) (softmax i -> MMA)
  const uint32_t bar_p_free = bar_p_full + 64;            // 2   PV_i(j) done: P_i free, O_i stable (MMA -> softmax i)
  const uint32_t bar_o_full = bar_p_free + 16;            // 2   last PV_i done               (MMA -> softmax i)
  const uint32_t tmem_slot = bar_o_full + 16;
  const uint32_t bar_v_zero = tmem_slot + 8;              // 1   V rows past seqlens zeroed (warp 3 -> MMA), MASKED only
  const uint32_t bar_v_tail = tmem_slot + 16;             // 1   softmax warp 4 reached the last KV tile (-> warp 3)
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + (tmem_slot - base));
  const uint32_t smem_q = base + Cfg::BAR_BYTES;                      // 2 Q tiles
  const uint32_t smem_k = smem_q + 2 * Cfg::Q_TILE_BYTES;             // STAGES K tiles
  const uint32_t smem_v = smem_k + STAGES * Cfg::KV_TILE_BYTES;       // STAGES V tiles

  // warp index via shuffle: the compiler then knows it is warp-uniform and keeps role code on the uniform datapath
  const uint32_t warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const uint32_t lane = threadIdx.x & 31;
  const int bh = blockIdx.y;
  // The masked build is a separate instantiation: the extra live values cost the unmasked D = 128 kernel (168 registers,
  // the cap at 384 threads) 56 bytes of spills and ~8 % when they were runtime flags of one kernel.
  const bool causal = MASKED && mask.causal;
  // causal: CTAs near the end of the sequence have the most KV tiles; start them first
  const int q0 = (causal ? int(gridDim.x - 1 - blockIdx.x) : int(blockIdx.x)) * 256;
  const int n_keys = (MASKED && mask.seqlens) ? min(N, max(1, mask.seqlens[bh / mask.H])) : N;  // valid keys of this batch
  const int Tk = (n_keys + BC - 1) / BC;
  const int T = causal ? min(Tk, (q0 + 256 + BC - 1) / BC) : Tk;  // KV tiles this CTA walks
  // Key padding: the last KV tile is loaded whole, so its keys in [seqlens[b], N) are real memory that TMA does not
  // zero-fill (it does past N).  Their P is exactly 0, but 0 * NaN / Inf in the PV product is NaN, so warp 3 zeroes those
  // V rows in shared memory and the MMA thread issues the PV products of that tile only after it has.  Warp 3 first waits
  // until softmax warp 4 reaches that tile: warp 4 has then seen PV_0 of tile T-3 complete, so every earlier use of the
  // V stage has landed and the parity wait on bar_v_full below cannot be satisfied by an older phase.
  const bool zero_v_tail = MASKED && n_keys < N && (n_keys % BC) != 0 && T == Tk;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 4; ++i) {
      mbar_init(bar_s_full + 8 * i, 1);
      mbar_init(bar_s_free + 8 * i, 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_q_full + 8 * i, 1);
      for (int p = 0; p < 4; ++p) mbar_init(bar_p_full + 32 * i + 8 * p, 4);
      mbar_init(bar_p_free + 8 * i, 1);
      mbar_init(bar_o_full + 8 * i, 1);
    }
    if (MASKED) {
      mbar_init(bar_v_zero, 32);
      mbar_init(bar_v_tail, 1);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_k_full + 8 * s, 1);
      mbar_init(bar_k_empty + 8 * s, 1);
      mbar_init(bar_v_full + 8 * s, 1);
      mbar_init(bar_v_empty + 8 * s, 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ---------------------------------------------------------------------------------- TMA producer
    // One lane is elected ONCE and runs the whole producer loop alone (waits included): per-batch elect + __syncwarp
    // and 32-lane barrier polling cost ~35 % of the tile time in tools/ubench/ubench_attn.cu; electing through
    // elect.sync (not `lane == 0`) keeps operands on the uniform datapath (no R2UR waterfall loops).
    if (elect_one()) {
      auto load_q = [&](int i) {
        const uint32_t bar = bar_q_full + 8 * i;
        {
          mbar_arrive_expect_tx(bar, Cfg::Q_TILE_BYTES);
#pragma unroll
          for (int c = 0; c < NCH; ++c)
            tma_load_3d(smem_q + i * Cfg::Q_TILE_BYTES + c * Cfg::Q_CHUNK_BYTES, &tmQ, bar, c * CW, q0 + i * 128, bh,
                        kPolicyEvictFirst);
        }
      };
      auto load_k = [&](int j) {
        const int s = j % STAGES;
        mbar_wait(bar_k_empty + 8 * s, ((j / STAGES) & 1) ^ 1);
        const uint32_t bar = bar_k_full + 8 * s;
        {
          mbar_arrive_expect_tx(bar, Cfg::KV_TILE_BYTES);
#pragma unroll
          for (int c = 0; c < NCH; ++c)
            tma_load_3d(smem_k + s * Cfg::KV_TILE_BYTES + c * Cfg::KV_CHUNK_BYTES, &tmK, bar, c * CW, j * BC, bh,
                        kPolicyEvictLast);
        }
      };
      auto load_v = [&](int j) {
        const int s = j % STAGES;
        mbar_wait(bar_v_empty + 8 * s, ((j / STAGES) & 1) ^ 1);
        const uint32_t bar = bar_v_full + 8 * s;
        const uint32_t dst = smem_v + s * Cfg::KV_TILE_BYTES;
        {
          mbar_arrive_expect_tx(bar, Cfg::KV_TILE_BYTES);
          if constexpr (Cfg::V_DN) {
            // V^T tile: D rows x BC keys, as [D rows x 64 keys] 128B-swizzled boxes (keys contiguous = K-major B operand)
#pragma unroll
            for (int c = 0; c < BC / 64; ++c)
              tma_load_3d(dst + c * (D * 128), &tmV, bar, j * BC + c * 64, 0, bh, kPolicyEvictLast);
          } else {
#pragma unroll
            for (int c = 0; c < NCH; ++c)
              tma_load_3d(dst + c * Cfg::KV_CHUNK_BYTES, &tmV, bar, c * CW, j * BC, bh, kPolicyEvictLast);
          }
        }
      };
      load_q(0);
      load_k(0);
      load_q(1);
      for (int j = 0; j < T; ++j) {
        if (j + 1 < T) load_k(j + 1);
        load_v(j);
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------------------------- MMA issuer
    // One lane is elected once and runs the whole issue loop (see the producer above).
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(128, BC, Cfg::DT, false, false);  // Q, K both K-major (D contiguous)
      // P from TMEM; V is MN-major ([keys, D], D contiguous) or, for V^T input, K-major ([D, keys], keys contiguous)
      constexpr uint32_t idesc_o = make_idesc(128, D, Cfg::DT, false, !Cfg::V_DN);
      constexpr uint64_t qk_hi = make_smem_desc_hi(16, 8 * ROWB, Cfg::SWZ_MODE);
      constexpr uint64_t v_hi = Cfg::V_DN ? make_smem_desc_hi(16, 1024, kSwizzle128B)
                                          : make_smem_desc_hi(Cfg::KV_CHUNK_BYTES, 8 * ROWB, Cfg::SWZ_MODE);
      constexpr int KSTEPS_PER_CHUNK = CW / 16;

      // S_i = Q_i K^T, then commit to `bar_a` (and optionally `bar_b`)
      auto issue_s = [&](int i, int stage, uint32_t bar_a, uint32_t bar_b) {
        const uint32_t q_addr = smem_q + i * Cfg::Q_TILE_BYTES;
        const uint32_t k_addr = smem_k + stage * Cfg::KV_TILE_BYTES;
        const uint32_t d_tmem = tmem_base + (i ? Cfg::S_COL1 : Cfg::S_COL0);
        {
#pragma unroll
          for (int k = 0; k < D / 16; ++k) {
            const uint32_t q_off = (k / KSTEPS_PER_CHUNK) * Cfg::Q_CHUNK_BYTES + (k % KSTEPS_PER_CHUNK) * 32;
            const uint32_t k_off = (k / KSTEPS_PER_CHUNK) * Cfg::KV_CHUNK_BYTES + (k % KSTEPS_PER_CHUNK) * 32;
            umma_ss<1>(d_tmem, smem_desc(qk_hi, q_addr + q_off), smem_desc(qk_hi, k_addr + k_off), idesc_s, k != 0);
          }
          umma_commit(bar_a);
          if (bar_b) umma_commit(bar_b);
        }
      };
      // O_i += P_i V.  P arrives in NP pieces of BC/NP keys (the softmax warps hand each piece over as soon as it is
      // written), so the first MMAs of PV_i(j) run under the exponentials of the later pieces.
      auto issue_pv = [&](int i, int stage, int j, uint32_t bar_a, uint32_t bar_b, uint32_t bar_c) {
        const uint32_t v_addr = smem_v + stage * Cfg::KV_TILE_BYTES;
        const uint32_t d_tmem = tmem_base + (i ? Cfg::O_COL1 : Cfg::O_COL0);
        const uint32_t p_tmem = tmem_base + (i ? Cfg::P_COL1 : Cfg::P_COL0);
        const bool accumulate = j > 0;
        {
#pragma unroll
          for (int k = 0; k < BC / 16; ++k) {
            if (k % (BC / 16 / NP) == 0) {
              if (k == 0 && zero_v_tail && j == Tk - 1) mbar_wait(bar_v_zero, 0);
              mbar_wait(bar_p_full + 32 * i + 8 * (k / (BC / 16 / NP)), j & 1);
              tc_fence_after();
              if (k == 0) tr(0, j, 5 + i);
            }
            // 16 keys = 8 packed fp16x2 columns of P; 16 rows of V = 16 * ROWB bytes (V^T: 32 bytes inside a 64-key box)
            const uint32_t v_off = Cfg::V_DN ? uint32_t((k / 4) * (D * 128) + (k % 4) * 32) : uint32_t(k * 16 * ROWB);
            umma_ts<1>(d_tmem, p_tmem + k * 8, smem_desc(v_hi, v_addr + v_off), idesc_o,
                       (accumulate || k != 0) ? 1u : 0u);
          }
          umma_commit(bar_a);
          if (bar_b) umma_commit(bar_b);
          if (bar_c) umma_commit(bar_c);
        }
      };

      mbar_wait(bar_q_full, 0);
      mbar_wait(bar_k_full, 0);
      tc_fence_after();
      issue_s(0, 0, bar_s_full, 0);
      mbar_wait(bar_q_full + 8, 0);
      tc_fence_after();
      if constexpr (Cfg::SHARE_S) {
        // One S buffer, the two tiles half a period apart.  Issue order per KV tile j (each step waits only for what it
        // needs, and in steady state the waits are satisfied in exactly this order):
        //   S_1(j)     once tile 0's warps hold S_0(j) in registers            (s_free0)
        //   PV_1(j-1)  as tile 1's P halves arrive                              (p_full1)
        //   S_0(j+1)   once tile 1's warps hold S_1(j) in registers            (s_free1)
        //   PV_0(j)    as tile 0's P halves arrive                              (p_full0)
        for (int j = 0; j < T; ++j) {
          const int s = j % STAGES, s1 = (j + 1) % STAGES, sp = (j + STAGES - 1) % STAGES;
          mbar_wait(bar_s_free, j & 1);
          tc_fence_after();
          issue_s(1, s, bar_s_full + 8, bar_k_empty + 8 * s);  // second and last reader of K(j)
          tr(0, j, 4);
          if (j > 0) {
            mbar_wait(bar_v_full + 8 * sp, ((j - 1) / STAGES) & 1);
            issue_pv(1, sp, j - 1, bar_p_free + 8, 0u, bar_v_empty + 8 * sp);
            tr(0, j, 3);
          }
          if (j + 1 < T) {
            mbar_wait(bar_k_full + 8 * s1, ((j + 1) / STAGES) & 1);
            mbar_wait(bar_s_free + 8, j & 1);
            tc_fence_after();
            issue_s(0, s1, bar_s_full, 0u);
            tr(0, j, 2);
          }
          mbar_wait(bar_v_full + 8 * s, (j / STAGES) & 1);
          issue_pv(0, s, j, bar_p_free, (j == T - 1) ? bar_o_full : 0u, 0u);
          tr(0, j, 1);
        }
        const int sl = (T - 1) % STAGES;
        issue_pv(1, sl, T - 1, bar_p_free + 8, bar_o_full + 8, bar_v_empty + 8 * sl);
      } else {
      issue_s(1, 0, bar_s_full + 8, bar_k_empty);
      for (int j = 0; j < T; ++j) {
        if constexpr (Cfg::ALIAS_P) {
          // P lives in the S columns: PV_i(j) first, then S_i(j+1) (in-order execution keeps P intact until read)
          const int s = j % STAGES;
          const int s1 = (j + 1) % STAGES;
          mbar_wait(bar_v_full + 8 * s, (j / STAGES) & 1);
          tr(0, j, 0);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            issue_pv(i, s, j, bar_p_free + 8 * i, (j == T - 1) ? bar_o_full + 8 * i : 0u,
                     i == 1 ? bar_v_empty + 8 * s : 0u);
            tr(0, j, 1 + 2 * i);
            if (j + 1 < T) {
              if (i == 0) {
                mbar_wait(bar_k_full + 8 * s1, ((j + 1) / STAGES) & 1);
                tc_fence_after();
              }
              issue_s(i, s1, bar_s_full + 8 * i, i == 1 ? bar_k_empty + 8 * s1 : 0u);
              tr(0, j, 2 + 2 * i);
            }
          }
          continue;
        }
        if (j + 1 < T) {
          // scores of the next KV tile: only needs the S columns back (the softmax warps hold tile j in registers)
          const int s1 = (j + 1) % STAGES;
          mbar_wait(bar_k_full + 8 * s1, ((j + 1) / STAGES) & 1);
          tr(0, j, 0);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            mbar_wait(bar_s_free + 8 * i, j & 1);
            tr(0, j, 1 + 2 * i);
            tc_fence_after();
            issue_s(i, s1, bar_s_full + 8 * i, i == 1 ? bar_k_empty + 8 * s1 : 0u);
            tr(0, j, 2 + 2 * i);
          }
        }
        const int s = j % STAGES;
        mbar_wait(bar_v_full + 8 * s, (j / STAGES) & 1);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          issue_pv(i, s, j, bar_p_free + 8 * i, (j == T - 1) ? bar_o_full + 8 * i : 0u,
                   i == 1 ? bar_v_empty + 8 * s : 0u);
        }
        tr(0, j, 7);
      }
      }
    }
  } else if (warp == 3) {
    if (zero_v_tail) {
      const int j = Tk - 1, s = j % STAGES;
      mbar_wait(bar_v_tail, 0);
      mbar_wait(bar_v_full + 8 * s, (j / STAGES) & 1);
      fa2_zero_v_keys<Cfg>(smem_v + s * Cfg::KV_TILE_BYTES, n_keys - j * BC, int(lane));
      mbar_arrive(bar_v_zero);
    }
  } else if (warp >= 4) {
    // ---------------------------------------------------------------------------------- softmax + epilogue
    const int i = (warp >= 8) ? 1 : 0;                  // which Q tile
    const uint32_t q = warp & 3;                         // TMEM lane quadrant
    const uint32_t lane_base = (q * 32) << 16;
    const uint32_t s_tmem = tmem_base + lane_base + (i ? Cfg::S_COL1 : Cfg::S_COL0);
    const uint32_t p_tmem = tmem_base + lane_base + (i ? Cfg::P_COL1 : Cfg::P_COL0);
    const uint32_t o_tmem = tmem_base + lane_base + (i ? Cfg::O_COL1 : Cfg::O_COL0);
    float m_ref = -INFINITY;  // reference max, in log2-scaled units
    float l = 0.f;
    // one KV tile of this row: scores in sr (fp32 bits) -> P (packed 16-bit pairs, in place) -> TMEM, statistics updated
    auto softmax_tile = [&](const int j, uint32_t* sr) {
      const bool tw = TRACE && lane == 0 && q == 0;  // one thread per warpgroup writes the trace
      float* s = reinterpret_cast<float*>(sr);
      if (j == Tk - 1 && (n_keys % BC) != 0) {
        // ragged last tile only.  The empty asm keeps this a real (warp-uniform) branch: if-converted, the 2 x BC
        // compare/select instructions would run on every tile.
        asm volatile("" ::: "memory");
        const int valid = n_keys - j * BC;
#pragma unroll
        for (int c = 0; c < BC; ++c)
          if (c >= valid) s[c] = -INFINITY;
      }
      if (MASKED && causal && (j + 1) * BC - 1 > q0 + i * 128 + int(q) * 32) {
        // this KV tile reaches past the diagonal for some row of the warp (warp-uniform test on the warp's first row)
        asm volatile("" ::: "memory");
        const int last = q0 + i * 128 + int(q) * 32 + int(lane) - j * BC;  // last visible key of this row, tile-relative
#pragma unroll
        for (int c = 0; c < BC; ++c)
          if (c > last) s[c] = -INFINITY;
      }
      const float mx = row_max<BC>(s) * scale_log2;
      // Has PV_i(j-1) been observed complete (O_i stable, P_i columns free)?  With ALIAS_P it always has: S_i(j) was
      // issued after PV_i(j-1) and tcgen05.commit covers all prior MMAs, so s_full(j) already implies it.
      bool pv_done = (j == 0) || Cfg::ALIAS_P;
      if (j == 0) {
        m_ref = mx;
      } else {
        const bool need = mx > m_ref + kRescaleThreshold;
        if (__any_sync(0xffffffffu, need)) {
          // warp-uniform: rescale this warp's 32 rows of O (rows that did not move use alpha = 1)
          if (!pv_done) {
            mbar_wait(bar_p_free + 8 * i, (j - 1) & 1);
            tc_fence_after();
            pv_done = true;
          }
          const float m_new = need ? mx : m_ref;
          const float alpha = fast_exp2(m_ref - m_new);
          m_ref = m_new;
          l *= alpha;
#pragma unroll
          for (int c = 0; c < D / 16; ++c) {  // 16-column pieces: the whole score row is live in registers here
            uint32_t orr[16];
            tmem_ld_32x32b_x16(o_tmem + c * 16, orr);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 16; ++e) orr[e] = __float_as_uint(__uint_as_float(orr[e]) * alpha);
            tmem_st_32x32b_x16(o_tmem + c * 16, orr);
          }
          tmem_wait_st();
        }
      }
      if (tw) tr(1 + i, j, 2);
      // P = exp2(s * scale_log2 - m_ref), row sum in fp32, P packed to fp16 pairs in place
      // processed in blocks of 16 with packed fp32x2 arithmetic (FFMA2 / FADD2: one issue slot per two elements);
      // all FFMA2s of a block, then its MUFU.EX2s, then sums / packs, so 16 independent exponentials are in flight
      float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
      const float neg_m = -m_ref;
      const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(neg_m, neg_m);
      constexpr int PIECE = BC / NP;  // keys per piece of P
#pragma unroll
      for (int c0 = 0; c0 < BC; c0 += 16) {
        float2 x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = ffma2(make_float2(s[c0 + 2 * e], s[c0 + 2 * e + 1]), scale2, negm2);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          // POLY of every 8 pairs are evaluated on the FMA/ALU pipes with packed fp32x2 arithmetic (no MUFU)
          const bool on_fma = (POLY == 1 && e == 3) || (POLY == 2 && (e == 2 || e == 6)) ||
                                  (POLY == 3 && (e == 2 || e == 5 || e == 7)) || (POLY == 4 && (e & 1));
          if (on_fma) {
            x[e] = exp2_poly3_x2(x[e]);
          } else {
            x[e].x = fast_exp2(x[e].x);
            x[e].y = fast_exp2(x[e].y);
          }
        }
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          acc0 = fadd2(acc0, x[e]);
          acc1 = fadd2(acc1, x[e + 1]);
          sr[(c0 >> 1) + e] = Cfg::DT == 1 ? pack_bf162(x[e].x, x[e].y) : pack_half2(x[e].x, x[e].y);
          sr[(c0 >> 1) + e + 1] = Cfg::DT == 1 ? pack_bf162(x[e + 1].x, x[e + 1].y) : pack_half2(x[e + 1].x, x[e + 1].y);
        }
        if ((c0 + 16) % PIECE == 0) {
          // piece complete: hand it to the MMA thread now, PV of this piece runs under the next piece's exponentials
          const int pc = c0 / PIECE;
          if (pc == 0 && !pv_done) {  // P_i(j-1) must have been consumed before it is overwritten (long since true)
            mbar_wait(bar_p_free + 8 * i, (j - 1) & 1);
            tc_fence_after();
          }
          if (tw && pc == 0) tr(1 + i, j, 3);
          tmem_st_n<PIECE / 2>(p_tmem + pc * (PIECE / 2), sr + pc * (PIECE / 2));
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_p_full + 32 * i + 8 * pc);
          if (tw && pc == 0) tr(1 + i, j, 4);
        }
      }
      l += (acc0.x + acc0.y) + (acc1.x + acc1.y);
      if (tw) tr(1 + i, j, 6);
    };
    for (int j = 0; j < T; ++j) {
      uint32_t sr[BC];
      const bool tw = TRACE && lane == 0 && q == 0;
      if (zero_v_tail && j == Tk - 1 && threadIdx.x == 128) mbar_arrive(bar_v_tail);
      mbar_wait(bar_s_full + 8 * i, j & 1);
      if (tw) tr(1 + i, j, 0);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < BC / 32; ++c) tmem_ld_32x32b_x32(s_tmem + c * 32, sr + c * 32);
      tmem_wait_ld();
      if (tw) tr(1 + i, j, 1);
      // the scores are in registers: give the S columns back so that S(j+1) is computed under this softmax
      if constexpr (!Cfg::ALIAS_P) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_s_free + 8 * i);
      }
      softmax_tile(j, sr);
    }
    // ---- epilogue: O_i / l -> fp16 -> swizzled smem (reusing this tile's Q buffer) -> TMA store
    mbar_wait(bar_o_full + 8 * i, 0);
    tc_fence_after();
    const float inv_l = 1.0f / l;
    const uint32_t stage_base = smem_q + i * Cfg::Q_TILE_BYTES + q * 32 * ROWB;  // this warp's 32 rows inside each chunk
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t orr[32];
      tmem_ld_32x32b_x32(o_tmem + c * 32, orr);
      tmem_wait_ld();
      const int chunk = (c * 32) / CW;
      const int sub0 = ((c * 32) % CW) / 8;  // first 16-byte piece inside the smem row
      const uint32_t row_addr = stage_base + chunk * Cfg::Q_CHUNK_BYTES + lane * ROWB;
      const uint32_t xr = (ROWB == 128) ? (lane & 7) : ((lane >> 1) & 3);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const float* f = reinterpret_cast<const float*>(orr + 8 * g);
        if constexpr (Cfg::DT == 1)
          st_shared_v4(row_addr + (((sub0 + g) ^ xr) << 4), pack_bf162(f[0] * inv_l, f[1] * inv_l),
                       pack_bf162(f[2] * inv_l, f[3] * inv_l), pack_bf162(f[4] * inv_l, f[5] * inv_l),
                       pack_bf162(f[6] * inv_l, f[7] * inv_l));
        else
          st_shared_v4(row_addr + (((sub0 + g) ^ xr) << 4), pack_half2(f[0] * inv_l, f[1] * inv_l),
                       pack_half2(f[2] * inv_l, f[3] * inv_l), pack_half2(f[4] * inv_l, f[5] * inv_l),
                       pack_half2(f[6] * inv_l, f[7] * inv_l));
      }
    }
    fence_proxy_async_smem();
    __syncwarp();
    const int row0 = q0 + i * 128 + int(q) * 32;
    if (lane == 0 && row0 < N) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) tma_store_3d(&tmO, stage_base + c * Cfg::Q_CHUNK_BYTES, c * CW, row0, bh);
      tma_store_commit();
      tma_store_wait_all<0>();
    }
    __syncwarp();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, Cfg::TMEM_COLS);
}

template <class Cfg>
static int launch_fa2(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N, float scale,
                      cudaStream_t stream, const DeviceInfo& di, int np = 0, bool trace = false, int poly = 0,
                      const Fa2Mask mask = Fa2Mask()) {
  constexpr int D = Cfg::D;
  const uint64_t BH = uint64_t(B) * uint64_t(H);
  CUtensorMap tmQ, tmK, tmV, tmO;
  int rc;
  if ((rc = make_tmap_3d_u16(&tmQ, Q, BH, N, D, uint64_t(N) * D, D, 1, 128, Cfg::CW, Cfg::ROWB))) return rc;
  if ((rc = make_tmap_3d_u16(&tmK, K, BH, N, D, uint64_t(N) * D, D, 1, Cfg::BC, Cfg::CW, Cfg::ROWB))) return rc;
  if (Cfg::V_DN) {
    if (N % 8)
      return set_error(B200K_EALIGN, "b200k_fa2_fwd_f16: V as [B,H,D,N] needs N %% 8 == 0 (16-byte rows), got N=%lld",
                       (long long)N);
    rc = make_tmap_3d_u16(&tmV, V, BH, D, N, uint64_t(N) * D, N, 1, D, 64, 128);
  } else {
    rc = make_tmap_3d_u16(&tmV, V, BH, N, D, uint64_t(N) * D, D, 1, Cfg::BC, Cfg::CW, Cfg::ROWB);
  }
  if (rc) return rc;
  if ((rc = make_tmap_3d_u16(&tmO, O, BH, N, D, uint64_t(N) * D, D, 1, 32, Cfg::CW, Cfg::ROWB))) return rc;
  dim3 grid(unsigned((N + 255) / 256), unsigned(BH));
  const float scale_log2 = scale * 1.4426950408889634f;
  using Kern = void (*)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, int, float,
                        unsigned long long*, const Fa2Mask);
  Kern kern;
  unsigned long long* tbuf = nullptr;
  // Experiment / debug instantiations (piece counts, cycle trace, higher polynomial fractions) only exist for the two
  // benchmark shapes; every configuration has the production pair (POLY 0 and 1, two pieces).
  constexpr bool kLab = (Cfg::D == 64 || Cfg::D == 128) && !Cfg::V_DN && Cfg::BC == 128 && Cfg::DT == 0;
  // Pieces per KV tile in which P is handed to the MMA thread.  With the shared S buffer PV is off the critical chain
  // and one hand-over per tile is best (D = 128: 1 -> 1267, 2 -> 1209, 4 -> 1202 TFLOP/s); otherwise two.
  constexpr int DEF_NP = Cfg::SHARE_S ? 1 : 2;
  constexpr int P2 = kLab ? 2 : 1, P3 = kLab ? 3 : 1, P4 = kLab ? 4 : 1;
  constexpr int NPA = kLab ? (DEF_NP == 1 ? 2 : 1) : DEF_NP, NPB = kLab ? 4 : DEF_NP;  // the two non-default counts
  constexpr bool TR = kLab;
  if (np == 0) np = DEF_NP;
  if (mask.causal || mask.seqlens) {
    kern = poly ? fa2_fwd_tcgen05_kernel<Cfg, false, 1, DEF_NP, true> : fa2_fwd_tcgen05_kernel<Cfg, false, 0, DEF_NP, true>;
  } else if (trace && g_fa2_trace && kLab) {
    tbuf = g_fa2_trace;
    kern = poly ? fa2_fwd_tcgen05_kernel<Cfg, TR, 1, DEF_NP> : fa2_fwd_tcgen05_kernel<Cfg, TR, 0, DEF_NP>;
  } else if (np != DEF_NP && kLab) {
    kern = np == 4 ? (poly ? fa2_fwd_tcgen05_kernel<Cfg, false, 1, NPB> : fa2_fwd_tcgen05_kernel<Cfg, false, 0, NPB>)
                   : (poly ? fa2_fwd_tcgen05_kernel<Cfg, false, 1, NPA> : fa2_fwd_tcgen05_kernel<Cfg, false, 0, NPA>);
  } else {
    kern = poly == 0   ? fa2_fwd_tcgen05_kernel<Cfg, false, 0, DEF_NP>
           : poly == 1 ? fa2_fwd_tcgen05_kernel<Cfg, false, 1, DEF_NP>
           : poly == 2 ? fa2_fwd_tcgen05_kernel<Cfg, false, P2, DEF_NP>
           : poly == 3 ? fa2_fwd_tcgen05_kernel<Cfg, false, P3, DEF_NP>
                       : fa2_fwd_tcgen05_kernel<Cfg, false, P4, DEF_NP>;
  }
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), di.device, Cfg::SMEM_BYTES)) return rc;
  kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(tmQ, tmK, tmV, tmO, int(N), scale_log2, tbuf, mask);
  B200K_CHECK_CUDA(cudaGetLastError());
  return B200K_OK;
}

}  // namespace b200k

extern "C" int b200k_fa2_fwd_f16(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N,
                                 int64_t D, float scale, int v_is_dn, int variant, void* stream) {
  return b200k_fa2_fwd(Q, K, V, O, B, H, N, D, scale, v_is_dn, B200K_F16, 0, nullptr, variant, stream);
}

extern "C" int b200k_fa2_fwd(const void* Q, const void* K, const void* V, void* O, int64_t B, int64_t H, int64_t N,
                             int64_t D, float scale, int v_is_dn, int dtype, int causal, const int* seqlens_k, int variant,
                             void* stream) {
  using namespace b200k;
  if (dtype != B200K_F16 && dtype != B200K_BF16)
    return set_error(B200K_EDTYPE, "b200k_fa2_fwd: dtype %d not supported (f16, bf16)", dtype);
  if (dtype == B200K_BF16 && v_is_dn)
    return set_error(B200K_EARG, "b200k_fa2_fwd: the [B,H,D,N] V layout is built for fp16 only");
  Fa2Mask mask;
  mask.seqlens = seqlens_k;
  mask.H = int(H);
  mask.causal = causal ? 1 : 0;
  const bool trace = (variant & 0x100) != 0;  // debugging: cycle trace of CTA (0,0), see b200k_debug_set_trace
  // Experiment switches (round-robin measurements on one B200, profiles/r01_fa2_variants.txt and r01_fa2_*.log;
  // TFLOP/s at (4,48,8192,64) unless noted):
  //   0x400        D = 128 only: P aliases S (S0 S1 O0 O1) instead of the shared S buffer: 1122 vs 1223.
  //   bits 12-13   P handed to the MMA thread in 1 / 2 / 4 pieces per KV tile.  D = 64: 731 / 817 / 761 -> 2;
  //                D = 128 (shared S): 1267 / 1209 / 1202 -> 1.
  //   bits 14-16   n of every 8 exponential pairs evaluated as a degree-3 polynomial on the FMA/ALU pipes instead
  //                of MUFU.EX2 (FlashAttention-4's trick): 0 -> 817, 1 -> 865, 2 -> 800, 3 -> 740, 4 -> 713;
  //                D = 128: 1144 / 1209 / 1155; D = 32: 414 / 426; D = 96: 912 / 920.  Default 1 (value 0), 7 = none.
  //   0x800        older spelling of "3 of 8".
  //   0x20000      D = 64 only: one shared S buffer as for D = 128 (forced ping-pong of the two tiles): 2 % slower.
  // Tried and removed (kept out of the build): exp2-phase turn-taking between the two softmax warpgroups through named
  // barriers (744 vs 812: a turn also holds the MUFU pipe through the P store / hand-over of the warpgroup that owns
  // it); two threads per query row (16 softmax warps, 96 registers): D = 64
  // 829 vs 799, D = 128 1217 vs 1211 - within noise for twice the softmax code; an event-driven MMA issue loop
  // (non-blocking mbarrier probes, whichever tile is ready): slower, the single issuing thread becomes the bottleneck.
  const int poly_sel = (variant >> 14) & 7;
  const int poly = poly_sel == 7 ? 0 : (poly_sel ? min(4, poly_sel) : ((variant & 0x800) ? 3 : 1));
  const int np_sel = (variant >> 12) & 3;  // 0 default, 1 -> 1 piece, 2 -> 2 pieces, 3 -> 4 pieces
  const int np = np_sel == 3 ? 4 : np_sel;  // 0 = the configuration's default
  if (!Q || !K || !V || !O) return set_error(B200K_EARG, "b200k_fa2_fwd: null pointer");
  if (B < 1 || H < 1 || N < 1 || N > INT32_MAX || B * H > 65535)
    return set_error(B200K_ESHAPE, "b200k_fa2_fwd_f16: need B,H,N >= 1 and B*H <= 65535 (got B=%lld H=%lld N=%lld)",
                     (long long)B, (long long)H, (long long)N);
  if (D != 32 && D != 64 && D != 96 && D != 128)
    return set_error(B200K_EHEADDIM, "headdim not support! (b200k_fa2_fwd_f16: D=%lld, supported 32/64/96/128)",
                     (long long)D);
  if (scale <= 0.f) scale = 1.0f / sqrtf(float(D));
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == B200K_BF16) {
    const int p01 = poly ? 1 : 0;  // the bf16 builds exist with the production exp2 settings only
    switch (D) {
      case 32: return launch_fa2<Fa2Cfg<32, 128, 4, false, false, false, 1>>(Q, K, V, O, B, H, N, scale, s, di, 0, false, p01, mask);
      case 64: return launch_fa2<Fa2Cfg<64, 128, 4, false, false, false, 1>>(Q, K, V, O, B, H, N, scale, s, di, 0, false, p01, mask);
      case 96: return launch_fa2<Fa2Cfg<96, 64, 4, false, false, false, 1>>(Q, K, V, O, B, H, N, scale, s, di, 0, false, p01, mask);
      default: return launch_fa2<Fa2Cfg<128, 128, 2, false, false, true, 1>>(Q, K, V, O, B, H, N, scale, s, di, 0, false, p01, mask);
    }
  }
  if (v_is_dn) {
    switch (D) {
      case 32: return launch_fa2<Fa2Cfg<32, 128, 4, true>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
      case 64: return launch_fa2<Fa2Cfg<64, 128, 4, true>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
      case 96: return launch_fa2<Fa2Cfg<96, 64, 4, true>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
      default: return launch_fa2<Fa2Cfg<128, 128, 2, true, false, true>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
    }
  }
  switch (D) {
    case 32: return launch_fa2<Fa2Cfg<32, 128, 4>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
    case 64:
      if (variant & 0x20000)  // one shared S buffer (forced ping-pong of the two tiles) as for D = 128: 2 % slower here
        return launch_fa2<Fa2Cfg<64, 128, 4, false, false, true>>(Q, K, V, O, B, H, N, scale, s, di, np, trace, poly, mask);
      return launch_fa2<Fa2Cfg<64, 128, 4>>(Q, K, V, O, B, H, N, scale, s, di, np, trace, poly, mask);
    case 96: return launch_fa2<Fa2Cfg<96, 64, 4>>(Q, K, V, O, B, H, N, scale, s, di, np, false, poly, mask);
    default:
      // 0x400: the older layout for D = 128 (P aliases S, S0 S1 O0 O1) instead of the shared S buffer
      if (variant & 0x400)
        return launch_fa2<Fa2Cfg<128, 128, 2, false, true>>(Q, K, V, O, B, H, N, scale, s, di, np, trace, poly, mask);
      return launch_fa2<Fa2Cfg<128, 128, 2, false, false, true>>(Q, K, V, O, B, H, N, scale, s, di, np, trace, poly, mask);
  }
}

// Debug hook (not part of the drop-in surface): device buffer of 3 * 32 * 8 uint64 that the next traced launch
// (variant | 0x100, D = 64 or 128) fills with clock64() stamps of CTA (0,0).
extern "C" int b200k_debug_set_trace(void* dev_u64_buffer) {
  b200k::g_fa2_trace = static_cast<unsigned long long*>(dev_u64_buffer);
  return B200K_OK;
}
