// Fused flash-style multi-head attention for sm_100a, second generation: head_dim 64, no mask, no dropout.
// Replaces  softmax((q * d^-0.5) k^T) v  of attention.py:53-59 (== xformers memory_efficient_attention, attention.py:74-77).
//
// What changed against attention.cuh (round 1: one 128-query tile per CTA, two CTAs per SM, every row shared by two
// threads; 0.37 ms at B=32 / N=1370 with the tensor pipe at 34 % and MUFU at 43 % -- latency bound, no pipe saturated):
//   * one PERSISTENT CTA per SM walks a list of work units; a unit = 256 queries (two 128-row tiles) of one (image, head),
//     so every K/V tile is fetched once per 256 queries and CTA start-up / TMEM allocation are paid once per launch;
//   * ONE thread per query row: softmax group t (4 warps) owns tile t, a thread holds its whole 128-column score row in
//     registers -- no row-maximum exchange through shared memory, no pair barriers;
//   * the two groups ping-pong on the tensor pipe: S_t(j+1) = Q_t K_{j+1}^T is issued as soon as group t has pulled S_t(j)
//     into registers, P_t(j) V_j as soon as the group has written P_t(j) to tensor memory; while one group runs its
//     exponentials (MUFU / FMA pipes) the other group's score tile and P V product occupy the tensor pipe;
//   * all 512 tensor-memory columns: S0 S1 (2 x 128 fp32), O0 O1 (2 x 64 fp32), P0 P1 (2 x 64 = 128 bf16 pairs).
//
//   warp 0      : TMA producer (Q_t once per unit, 3-stage K ring, 3-stage V ring), whole warp converged, elected lane
//   warp 2      : tcgen05 issuer of the score tiles S_t = Q_t K^T (both query tiles)
//   warps 1, 3  : tcgen05 issuers of O_t += P_t V for tile 0 / tile 1 (warp 1 also allocates tensor memory)
//                 (all issuers run converged with one elected lane per instruction; three warps on three schedulers because
//                 a single issuing warp was the bottleneck, see below)
//   warps 4..7  : softmax group 0 (query tile 0)      warps 8..11 : softmax group 1 (query tile 1)
// Registers: compiled for 168 per thread (3 warps per scheduler); the control warpgroup drops to 72 and the softmax
// warpgroups take 216 each (setmaxnreg), enough for a 128-column fp32 score row per thread without spills.
//
// Hand-offs: tcgen05.commit -> mbarrier for everything the tensor pipe produces (S ready, P V retired, smem slots free);
// hardware named barriers (bar.arrive by the 128 group threads, bar.sync by the issuer warp) for "S is in registers" and
// "P is in tensor memory" -- tens of cycles instead of an mbarrier round trip.
// The running output stays in tensor memory across KV tiles, kept relative to a *stale* row maximum: O is only rescaled
// (tcgen05.ld -> scale -> tcgen05.st by the owning thread) when some row maximum of the warp grows by more than 2^8.
#pragma once
#include "ptx.cuh"

namespace ada {

constexpr int kFaThreads = 384;        // one thread per score row
constexpr int kFaThreadsSplit = 640;   // SPLIT: two threads per score row (16 softmax warps)
constexpr int kFaStages = 3;                       // K ring and V ring depth
constexpr int kFaTile = 128 * 64 * 2;              // one 128 x 64 bf16 tile: 16 KB
constexpr int kFaOffK = 2 * kFaTile;               // after Q0, Q1
constexpr int kFaOffV = kFaOffK + kFaStages * kFaTile;
constexpr int kFaOffO = kFaOffV + kFaStages * kFaTile;   // two output staging tiles
constexpr int kFaOffBar = kFaOffO + 2 * kFaTile;
constexpr int kFaOffXch = kFaOffBar + 256;                // SPLIT: row-maximum / row-sum exchange of the two row owners
constexpr int kFaSmemBytes = kFaOffXch + 6144;
constexpr int kFaTmemCols = 512;
constexpr float kFaRescaleLog2 = 8.0f;             // rescale O only when a row max grows by more than 2^8

struct FaArgs {
  int B, N, heads, D;        // D = heads * 64
  int units_per_seq;         // ceil(ceil(N / 128) / 2): 256-query units per (image, head)
  int total_units;           // B * heads * units_per_seq
  float scale_log2e;         // d^-0.5 * log2(e)
};

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// bit p set = exponential pair p (of every 16) runs on the FMA pipe; EMU of 16, evenly spaced
__host__ __device__ constexpr uint32_t fa_emu_mask(int emu) {
  if (emu < 0) return 0u;
  if (emu == 6) return 0x9249u;  // the pattern attention.cuh uses: both kernels then produce bit-identical results
  uint32_t m = 0;
  for (int p = 0; p < 16; ++p)
    if ((p * emu) % 16 < emu) m |= 1u << p;
  return m;
}

template <bool B>
struct FaTag {
  static constexpr bool value = B;
};

// Work unit idx -> (image, head, first query). Units of one image are adjacent (its K/V stay in L2: 16 heads x 350 KB) and
// inside an image the unit index is the slow one, so the short last unit of every head (N = 1370: 90 rows, one tile) is
// spread evenly over the persistent CTAs (consecutive CTAs take consecutive heads of the same unit index).
struct FaUnit {
  int img, head, q0;
  bool valid[2];
};
__device__ __forceinline__ FaUnit fa_unit(int idx, const FaArgs& a) {
  FaUnit u;
  if (idx >= a.total_units) {
    u.img = u.head = u.q0 = 0;
    u.valid[0] = u.valid[1] = false;
    return u;
  }
  const int per_img = a.heads * a.units_per_seq;
  u.img = idx / per_img;
  const int r = idx - u.img * per_img;
  const int uq = r / a.heads;
  u.head = r - uq * a.heads;
  u.q0 = uq * 256;
  u.valid[0] = true;
  u.valid[1] = u.q0 + 128 < a.N;
  return u;
}

// EMU = how many of every 16 exponential pairs are evaluated on the FMA pipe (Cody-Waite + degree-3 polynomial) instead of
// MUFU.EX2; the kernel is MUFU-bound at head_dim 64 (128 x 128 exponentials per 128-key tile = 1024 MUFU cycles per SM
// against 512 cycles of MMA), so the split between the two pipes is the tuning knob.
// SPLIT: every score row is shared by two threads (64 columns each), 16 softmax warps per CTA = 4 per scheduler, exactly
// the per-thread arithmetic of attention.cuh (bit-identical results) inside this kernel's persistent two-tile frame. The
// timing skeleton of the one-thread-per-row version (exponentials replaced by a copy) runs in 0.25 ms of 0.37 ms: with two
// softmax warps per scheduler a warp's phases (wait, tcgen05.ld, maximum, exponentials, tcgen05.st) are simply serialised;
// four warps per scheduler let one warp's exponentials (MUFU) overlap the others' fixed-latency phases.
// Measured (B200, 32 x 1370 x 16 heads): 0.393 ms, against 0.360 ms for one thread per row and 0.350 ms for attention.cuh;
// bit-identical to both (tools/gpu_check.py attention_geo_*). The pair exchange through shared memory and the 104
// register cap (a few spills in the exponential loop) cost more than the extra warps hide; kept as impl = 2 for the record.
template <int EMU, bool STAGGER, int WAITP, bool SPLIT = false>
__global__ void __launch_bounds__(SPLIT ? kFaThreadsSplit : kFaThreads, 1)
attention_fa_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_out,
                    const FaArgs a) {
  extern __shared__ __align__(1024) uint8_t fa_smem[];
  const uint32_t sbase = smem_u32(fa_smem);
  const uint32_t bar = sbase + kFaOffBar;
  auto q_full = [&](int t) { return bar + 8u * t; };
  auto q_free = [&](int t) { return bar + 8u * (2 + t); };
  auto s_full = [&](int t) { return bar + 8u * (4 + t); };
  auto o_full = [&](int t) { return bar + 8u * (6 + t); };   // one completion per retired P_t V product
  auto o_free = [&](int t) { return bar + 8u * (8 + t); };   // the epilogue of group t has read O_t out of tensor memory
  auto k_full = [&](int s) { return bar + 8u * (10 + s); };
  auto k_free = [&](int s) { return bar + 8u * (13 + s); };
  auto v_full = [&](int s) { return bar + 8u * (16 + s); };
  auto v_free = [&](int s) { return bar + 8u * (19 + s); };
  const uint32_t tmem_ptr_smem = bar + 8u * 22;
  // named barriers: 1 + t "S_t is in registers", 3 + t "P_t is in tensor memory" (128 group threads arrive, the issuer
  // warp syncs), 5 + t group-internal (epilogue staging)
  // 7: stagger. Both groups share the MUFU and FMA pipes of their schedulers; started together they run their exponential
  // phases at the same time (each at half rate) and then leave the pipes idle together. Group 1 therefore starts every
  // unit only once group 0 is half way through the exponentials of its first tile; the offset then persists.
  constexpr int kBarSL = 1, kBarPF = 3, kBarWG = SPLIT ? 13 : 5, kBarStagger = 7;
  constexpr int kBarPair = 5;                       // SPLIT: 5 + 4 * tile + lane quarter: the two warps that share 32 rows
  constexpr int kGroupSync = (SPLIT ? 256 : 128) + 32;  // softmax threads of one tile + the issuing warp

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kv = (a.N + 127) / 128;
  const bool ragged = (a.N & 127) != 0;

  if (threadIdx.x == 0) {
    if (sbase & 1023u) {  // the swizzled layouts below assume a 1 KB aligned window
      g_dev_error[0] = 0xA12;
      __trap();
    }
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_out);
    for (int t = 0; t < 2; ++t) {
      mbar_init(q_full(t), 1);
      mbar_init(q_free(t), 1);
      mbar_init(s_full(t), 1);
      mbar_init(o_full(t), 1);
      mbar_init(o_free(t), SPLIT ? 8 : 4);  // one arrival per warp of the group
    }
    for (int s = 0; s < kFaStages; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(k_free(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(v_free(s), 2);  // one arrival per P V issuer (tile)
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, kFaTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  griddep_wait();  // (programmatic dependent launch) everything above overlapped the previous kernel's tail
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_smem));

  if (warp < 4) {
  if constexpr (SPLIT) asm volatile("setmaxnreg.dec.sync.aligned.u32 56;"); else asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
  if (warp == 0) {
    // ------------------------------------------------------------------ producer (whole warp, elected lane per instruction)
    uint32_t qph[2] = {0u, 0u};
    int ks = 0, vs = 0;
    uint32_t kph = 0, vph = 0;
    for (int idx = blockIdx.x; idx < a.total_units; idx += gridDim.x) {
      if (idx + static_cast<int>(gridDim.x) >= a.total_units) griddep_launch_dependents();  // this CTA is on its last unit
      const FaUnit u = fa_unit(idx, a);
      auto load_q = [&](int t) {
        mbar_wait(q_free(t), qph[t] ^ 1u, 0x600 + t);  // every S MMA that reads the previous unit's Q_t has been issued and retired
        qph[t] ^= 1u;
        mbar_expect_tx_w(q_full(t), kFaTile);
        tma_load_3d_w(sbase + t * kFaTile, &tmap_qkv, q_full(t), u.head * 64, u.q0 + 128 * t, u.img);
      };
      auto load_k = [&](int j) {
        mbar_wait(k_free(ks), kph ^ 1u, 0x610 + ks);
        mbar_expect_tx_w(k_full(ks), kFaTile);
        tma_load_3d_w(sbase + kFaOffK + ks * kFaTile, &tmap_qkv, k_full(ks), a.D + u.head * 64, j * 128, u.img);
        if (++ks == kFaStages) { ks = 0; kph ^= 1u; }
      };
      auto load_v = [&](int j) {
        mbar_wait(v_free(vs), vph ^ 1u, 0x620 + vs);
        mbar_expect_tx_w(v_full(vs), kFaTile);
        tma_load_3d_w(sbase + kFaOffV + vs * kFaTile, &tmap_qkv, v_full(vs), 2 * a.D + u.head * 64, j * 128, u.img);
        if (++vs == kFaStages) { vs = 0; vph ^= 1u; }
      };
      load_q(0);
      load_k(0);
      if (u.valid[1]) load_q(1);
      load_v(0);
      for (int j = 1; j < num_kv; ++j) {
        load_k(j);
        load_v(j);
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ score issuer: S_t = Q_t K^T for both tiles
    // Three issuing warps on three different schedulers (this one, and one P V issuer per tile): a tcgen05.mma shares the
    // scheduler's MIO queue with the MUFU instructions of the two softmax warps that live there and takes ~100 cycles to
    // get through it (clock64 timelines, profiles/README.md); with all 24 MMAs of a 256-query x 128-key step issued by
    // one warp the ISSUER was the bottleneck (24 x ~105 cycles = the whole step), in this kernel and in attention.cuh.
    constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
    const uint64_t dq0 = make_smem_desc_sw128(sbase, 16, 1024);
    const uint64_t dk0 = make_smem_desc_sw128(sbase + kFaOffK, 16, 1024);
    uint32_t qfp[2] = {0u, 0u};
    int ks = 0;
    uint32_t kph = 0;
    // S_t(jj) = Q_t K_jj^T of unit `U` for both tiles; sync_t: first wait until group t has pulled its previous score
    // tile into registers (the tensor-memory columns are about to be overwritten).
    auto issue_s = [&](const FaUnit& U, int jj, bool sync0, bool sync1) {
      bool kwaited = false;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        if (t == 0 ? sync0 : sync1) named_bar_sync(kBarSL + t, kGroupSync);
        if (!U.valid[t]) continue;
        if (jj == 0) {
          mbar_wait(q_full(t), qfp[t], 0x630 + t);
          qfp[t] ^= 1u;
        }
        if (!kwaited) {
          mbar_wait(k_full(ks), kph, 0x640 + ks);
          kwaited = true;
        }
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + 128u * t;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_ss_w(d_tmem, dq0 + t * (kFaTile >> 4) + 2 * k, dk0 + ks * (kFaTile >> 4) + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        umma_commit_w(s_full(t));
        if (jj == num_kv - 1) umma_commit_w(q_free(t));  // last read of this unit's Q_t
      }
      if (kwaited) {
        umma_commit_w(k_free(ks));
        if (++ks == kFaStages) { ks = 0; kph ^= 1u; }
      }
    };
    int idx = blockIdx.x;
    FaUnit cur = fa_unit(idx, a);
    if (cur.valid[0]) issue_s(cur, 0, false, false);
    while (cur.valid[0]) {
      idx += gridDim.x;
      const FaUnit nxt = fa_unit(idx, a);
      for (int j = 0; j < num_kv; ++j) {
        if (j + 1 < num_kv)
          issue_s(cur, j + 1, cur.valid[0], cur.valid[1]);
        else
          issue_s(nxt, 0, cur.valid[0], cur.valid[1]);  // the next unit's first score tiles start under this unit's tail
      }
      cur = nxt;
    }
  } else {
    // ------------------------------------------------------------------ P V issuers: warp 1 -> tile 0, warp 3 -> tile 1
    // O_t (+)= P_t(j) V_j. Each V slot is released by two arrivals (one per tile); in a unit without a second tile the
    // tile-0 issuer provides both and the tile-1 issuer only keeps its ring position.
    const int t = (warp == 1) ? 0 : 1;
    constexpr uint32_t idesc_o = make_idesc_bf16(128, 64, 0, 1);  // B = V is MN-major (d contiguous)
    const uint64_t dv0 = make_smem_desc_sw128(sbase + kFaOffV, 0, 1024);
    const uint32_t d_tmem = tmem_base + 256u + 64u * t;
    const uint32_t p_tmem = tmem_base + 384u + 64u * t;
    uint32_t ofp = 0;
    int vs = 0;
    uint32_t vph = 0;
    for (int idx = blockIdx.x; idx < a.total_units; idx += gridDim.x) {
      const FaUnit u = fa_unit(idx, a);
      if (!u.valid[t]) {  // (tile 1 of a short unit) walk the ring without touching it
        for (int j = 0; j < num_kv; ++j)
          if (++vs == kFaStages) { vs = 0; vph ^= 1u; }
        continue;
      }
      for (int j = 0; j < num_kv; ++j) {
        named_bar_sync(kBarPF + t, kGroupSync);  // P_t(j) is in tensor memory (and O_t rescaled if it had to be)
        mbar_wait(v_full(vs), vph, 0x650 + vs);
        if (j == 0) {  // the previous unit's epilogue must have read O_t before it is overwritten
          mbar_wait(o_free(t), ofp ^ 1u, 0x660 + t);
          ofp ^= 1u;
        }
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)  // 16 keys per MMA = 8 packed tensor-memory columns of P
          umma_bf16_ts_w(d_tmem, p_tmem + kk * 8, dv0 + vs * (kFaTile >> 4) + kk * 128, idesc_o, (j > 0 || kk > 0) ? 1u : 0u);
        umma_commit_w(o_full(t));
        umma_commit_w(v_free(vs));
        if (!u.valid[1]) umma_commit_w(v_free(vs));  // (t == 0 here) the absent tile's arrival
        if (++vs == kFaStages) { vs = 0; vph ^= 1u; }
      }
    }
  }
  } else if constexpr (SPLIT) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // ------------------------------------------------------------------ softmax groups, two threads per query row
    const int w8 = warp - 4;
    const int t = w8 >> 3;                 // group = query tile (8 warps each)
    const int half = (w8 >> 2) & 1;        // which 64 score columns of the row this thread owns
    const int qd = warp & 3;               // tensor-memory lane quarter this warp may access
    const int row = qd * 32 + lane;
    const int gthread = threadIdx.x - 128 - 256 * t;  // 0..255 within the group
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const uint32_t tS = tmem_base + 128u * t + lane_off + 64u * half;
    const uint32_t tO = tmem_base + 256u + 64u * t + lane_off + 32u * half;
    const uint32_t tP = tmem_base + 384u + 64u * t + lane_off + 32u * half;
    const uint32_t sO = sbase + kFaOffO + t * kFaTile;
    float* xm = reinterpret_cast<float*>(fa_smem + kFaOffXch) + t * 768;  // [2 parities][2 halves][128 rows] row maxima
    float* xl = xm + 512;                                                  // [2 halves][128 rows] row sums
    const int pair_bar = kBarPair + 4 * t + qd;
    const float c = a.scale_log2e;
    uint32_t sfp = 0, ofp = 0;
    bool stored = false;

    for (int idx = blockIdx.x; idx < a.total_units; idx += gridDim.x) {
      const FaUnit u = fa_unit(idx, a);
      if (!u.valid[t]) continue;
      float m_used = -INFINITY, l_part = 0.f;
      auto tile = [&](const int j, auto masked_tag) {
        constexpr bool MASKED = decltype(masked_tag)::value;
        mbar_wait(s_full(t), sfp, 0x670 + t);
        sfp ^= 1u;
        tc_fence_after();
        uint32_t s0[32], s1[32];
        tmem_ld32(tS, s0);
        tmem_ld32(tS + 32, s1);
        tmem_ld_wait();
        tc_fence_before();
        named_bar_arrive(kBarSL + t, kGroupSync);  // S_t(j) lives in registers: the issuer may overwrite it with S_t(j+1)
        if constexpr (MASKED) {  // ragged last tile: keys past N are zero-filled by TMA -> mask them out
          const int kv_valid = min(128, a.N - j * 128) - half * 64;  // valid keys inside this thread's 64 columns
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (i >= kv_valid) s0[i] = 0xff800000u;
            if (32 + i >= kv_valid) s1[i] = 0xff800000u;
          }
        }
        float tm[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t* v = (k < 2) ? (s0 + 16 * k) : (s1 + 16 * (k - 2));
          float x = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
#pragma unroll
          for (int i = 3; i < 15; i += 2) x = fmax3(x, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          tm[k] = fmaxf(x, __uint_as_float(v[15]));
        }
        float tmax = fmaxf(fmaxf(tm[0], tm[1]), fmaxf(tm[2], tm[3]));
        // the two owners of a row combine their partial maxima (double-buffered by tile parity)
        float* xmj = xm + (j & 1) * 256;
        xmj[half * 128 + row] = tmax;
        named_bar_sync(pair_bar, 64);
        tmax = fmaxf(tmax, xmj[(half ^ 1) * 128 + row]);
        float sc = 1.0f;
        bool rescale = false;
        if (j == 0) {
          m_used = tmax;
        } else {
          const bool grow = (tmax - m_used) * c > kFaRescaleLog2;
          rescale = __any_sync(0xffffffffu, grow);  // rare; identical in both warps of the pair (same combined maxima)
          if (rescale) {
            const float m_new = fmaxf(m_used, tmax);
            sc = fast_exp2((m_used - m_new) * c);
            m_used = m_new;
            l_part *= sc;
            mbar_wait(o_full(t), ofp, 0x680 + t);  // P_t(j-1) V_{j-1} must have retired before O_t may be rescaled
            tc_fence_after();
#pragma unroll 1
            for (int h = 0; h < 4; ++h) {  // this thread's 32 of the row's 64 accumulator columns
              uint32_t r[8];
              tmem_ld8(tO + h * 8, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 8; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * sc);
              tmem_st8(tO + h * 8, r);
            }
          }
        }
        const float mc = m_used * c;
        constexpr uint32_t kEmuMask = fa_emu_mask(EMU);
        const uint64_t c2 = f2_pack(c, c), nmc2 = f2_pack(-mc, -mc);
        uint64_t rs2[4] = {0ull, 0ull, 0ull, 0ull};
        uint32_t pk[32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const uint64_t x2 = f2_fma(f2_pack(__uint_as_float(h ? s1[i] : s0[i]), __uint_as_float(h ? s1[i + 1] : s0[i + 1])), c2, nmc2);
            float p0, p1;
            if ((kEmuMask >> (i >> 1)) & 1u) {
              exp2_fma2(x2, p0, p1);
            } else {
              float x0, x1;
              f2_unpack(x2, x0, x1);
              p0 = fast_exp2(x0);
              p1 = fast_exp2(x1);
            }
            rs2[(i >> 1) & 3] = f2_add(rs2[(i >> 1) & 3], f2_pack(p0, p1));
            pk[h * 16 + (i >> 1)] = pack_bf16x2(p0, p1);
          }
        }
        {
          float a0, a1;
          f2_unpack(f2_add(f2_add(rs2[0], rs2[1]), f2_add(rs2[2], rs2[3])), a0, a1);
          l_part += a0 + a1;
        }
        if (j > 0) {  // P_t(j-1) V_{j-1} must have retired before P_t is overwritten (issued a whole tile ago)
          if (!rescale) mbar_wait(o_full(t), ofp, 0x680 + t);
          ofp ^= 1u;
          tc_fence_after();
        }
        tmem_st32(tP, pk);
        tmem_st_wait();
        tc_fence_before();
        named_bar_arrive(kBarPF + t, kGroupSync);  // P_t(j) is in tensor memory
      };
#pragma unroll 1
      for (int j = 0; j < num_kv - 1; ++j) tile(j, FaTag<false>{});
      if (ragged)
        tile(num_kv - 1, FaTag<true>{});
      else
        tile(num_kv - 1, FaTag<false>{});
      // ---- epilogue
      xl[half * 128 + row] = l_part;
      mbar_wait(o_full(t), ofp, 0x690 + t);  // the last P V of this unit has retired
      ofp ^= 1u;
      tc_fence_after();
      named_bar_sync(pair_bar, 64);
      const float inv = 1.0f / (l_part + xl[(half ^ 1) * 128 + row]);
      uint32_t o[32];
      tmem_ld32(tO, o);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free(t));  // O_t may be overwritten by the next unit's first P V
      if (gthread == 0 && stored) bulk_wait_read<0>();  // the previous unit's store has finished reading the staging tile
      named_bar_sync(kBarWG + t, 256);
      const uint32_t o_row = sO + static_cast<uint32_t>(row) * 128u;
      const uint32_t o_sw = static_cast<uint32_t>(row & 7);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t chunk = static_cast<uint32_t>(half * 4 + i);
        st_shared_v4(o_row + ((chunk ^ o_sw) << 4),
                     pack_bf16x2(__uint_as_float(o[8 * i]) * inv, __uint_as_float(o[8 * i + 1]) * inv),
                     pack_bf16x2(__uint_as_float(o[8 * i + 2]) * inv, __uint_as_float(o[8 * i + 3]) * inv),
                     pack_bf16x2(__uint_as_float(o[8 * i + 4]) * inv, __uint_as_float(o[8 * i + 5]) * inv),
                     pack_bf16x2(__uint_as_float(o[8 * i + 6]) * inv, __uint_as_float(o[8 * i + 7]) * inv));
      }
      fence_proxy_async_smem();
      named_bar_sync(kBarWG + t, 256);
      if (gthread == 0) {
        tma_store_3d(&tmap_out, sO, u.head * 64, u.q0 + 128 * t, u.img);
        bulk_commit();
        stored = true;
      }
    }
    if (gthread == 0 && stored) bulk_wait<0>();
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    // ------------------------------------------------------------------ softmax groups (one thread = one query row)
    const int t = (warp - 4) >> 2;         // group = query tile
    const int qd = warp & 3;               // tensor-memory lane quarter this warp may access
    const int row = qd * 32 + lane;
    const int gthread = threadIdx.x - 128 - 128 * t;  // 0..127 within the group
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const uint32_t tS = tmem_base + 128u * t + lane_off;
    const uint32_t tO = tmem_base + 256u + 64u * t + lane_off;
    const uint32_t tP = tmem_base + 384u + 64u * t + lane_off;
    const uint32_t sO = sbase + kFaOffO + t * kFaTile;
    const float c = a.scale_log2e;
    uint32_t sfp = 0, ofp = 0;
    bool stored = false;  // (group thread 0) a TMA store of this group's staging tile may still be reading it

    for (int idx = blockIdx.x; idx < a.total_units; idx += gridDim.x) {
      const FaUnit u = fa_unit(idx, a);
      if (!u.valid[t]) continue;
      float m_used = -INFINITY, l_sum[2] = {0.f, 0.f};
      if (STAGGER && t == 1) named_bar_sync(kBarStagger, 256);

      // One KV tile. MASKED (compile-time): only the ragged last tile carries the 128 compare+select pairs that overwrite
      // the scores of keys past N (zero-filled by TMA) with -inf.
#ifdef ADA_BRINGUP
      // clock64 timeline of lane 0 of the first warp of each group (CTA 0, first two units): 7 stamps per tile at
      // g_dev_timeline[t * 154 + tile * 7 + k]; the issuer's 9 stamps per iteration follow at 308 (ada_debug_timeline)
      const bool tl = blockIdx.x == 0 && qd == 0 && lane == 0 && idx < static_cast<int>(2 * gridDim.x);
      const int tl_base = t * 154 + (idx >= static_cast<int>(gridDim.x) ? num_kv * 7 : 0);
      auto stamp = [&](int j, int k) {
        if (tl && j < 11) g_dev_timeline[tl_base + j * 7 + k] = clock64();
      };
#else
      auto stamp = [](int, int) {};
#endif
      auto tile = [&](const int j, auto masked_tag) {
        constexpr bool MASKED = decltype(masked_tag)::value;
        stamp(j, 0);
        mbar_wait(s_full(t), sfp, 0x670 + t);
        stamp(j, 1);
        sfp ^= 1u;
        tc_fence_after();
        uint32_t s[4][32];
#pragma unroll
        for (int q = 0; q < 4; ++q) tmem_ld32(tS + 32 * q, s[q]);
        tmem_ld_wait();
        stamp(j, 2);
        tc_fence_before();
        named_bar_arrive(kBarSL + t, kGroupSync);  // S_t(j) lives in registers: the issuer may overwrite it with S_t(j+1)
        const int kv_valid = MASKED ? a.N - j * 128 : 128;  // keys of this tile that exist
        if constexpr (MASKED) {
          // only the 32-column chunks that straddle or lie past N pay for the compare+select pairs (warp-uniform branch)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int v = kv_valid - 32 * q;
            if (v < 32) {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (i >= v) s[q][i] = 0xff800000u;
            }
          }
        }
        float tm[8];  // FMNMX3: two scores per instruction, eight independent chains of 16 scores (dependent depth 8)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint32_t* v = &s[q >> 1][(q & 1) * 16];
          float x = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
#pragma unroll
          for (int i = 3; i < 15; i += 2) x = fmax3(x, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          tm[q] = fmaxf(x, __uint_as_float(v[15]));
        }
        const float tmax = fmax3(fmax3(tm[0], tm[1], tm[2]), fmax3(tm[3], tm[4], tm[5]), fmaxf(tm[6], tm[7]));
        // ---- running (stale) maximum; the decision to rescale is taken per warp
        float sc = 1.0f;
        bool rescale = false;
        if (j == 0) {
          m_used = tmax;
        } else {
          const bool grow = (tmax - m_used) * c > kFaRescaleLog2;
          rescale = __any_sync(0xffffffffu, grow);  // rare (first tile or two)
          stamp(j, 3);
          if (rescale) {
            const float m_new = fmaxf(m_used, tmax);
            sc = fast_exp2((m_used - m_new) * c);
            m_used = m_new;
            l_sum[0] *= sc;
            l_sum[1] *= sc;
          }
          if (rescale || WAITP == 0) {
            // P_t(j-1) V_{j-1} must have retired before O_t may be rescaled (WAITP == 0: and before P_t is overwritten)
            mbar_wait(o_full(t), ofp, 0x680 + t);
            tc_fence_after();
          }
          if (rescale) {
#pragma unroll 1
            for (int h = 0; h < 8; ++h) {
              uint32_t r[8];
              tmem_ld8(tO + h * 8, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 8; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * sc);
              tmem_st8(tO + h * 8, r);
            }
          }
        }
        stamp(j, 4);
        const float mc = m_used * c;
        // exponentials, row sum, bf16 pack; 32 columns at a time so that each quarter of P goes to tensor memory as soon as
        // it exists (16 packed columns) and the score registers die progressively
        constexpr uint32_t kEmuMask = fa_emu_mask(EMU);
        const uint64_t c2 = f2_pack(c, c), nmc2 = f2_pack(-mc, -mc);
        // independent packed row-sum chains, kept apart for columns 0..63 and 64..127: the same summation order as the two
        // threads that share a row in attention.cuh, so that the two kernels agree bit for bit (an image must not change
        // with the batch size it is processed in, and the kernel is selected by grid size)
        uint64_t rs2[2][4] = {{0ull, 0ull, 0ull, 0ull}, {0ull, 0ull, 0ull, 0ull}};
        uint32_t pk[4][16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (MASKED && kv_valid <= 32 * q) {  // (ragged last tile) a chunk entirely past N: P = 0, no exponentials
#pragma unroll
            for (int i = 0; i < 16; ++i) pk[q][i] = 0u;
          } else {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const uint64_t x2 = f2_fma(f2_pack(__uint_as_float(s[q][i]), __uint_as_float(s[q][i + 1])), c2, nmc2);
            float p0, p1;
            if constexpr (EMU == -1) {  // (bring-up) timing skeleton: exponentials replaced by a copy, wrong results
              f2_unpack(x2, p0, p1);
            } else if constexpr (EMU == -2) {  // (bring-up) skeleton without any per-element arithmetic but the pack
              p0 = __uint_as_float(s[q][i]);
              p1 = __uint_as_float(s[q][i + 1]);
            } else if ((kEmuMask >> (i >> 1)) & 1u) {
              exp2_fma2(x2, p0, p1);
            } else {
              float x0, x1;
              f2_unpack(x2, x0, x1);
              p0 = fast_exp2(x0);
              p1 = fast_exp2(x1);
            }
            if constexpr (EMU != -2) rs2[q >> 1][(i >> 1) & 3] = f2_add(rs2[q >> 1][(i >> 1) & 3], f2_pack(p0, p1));
            pk[q][i >> 1] = pack_bf16x2(p0, p1);
          }
          }
          // P_t(j-1) V_{j-1} must have retired before P_t is overwritten. WAITP: 0 = waited before the exponentials (above),
          // 1 = after the first quarter of them, 2 = after all of them (the four stores then go out back to back)
          if (WAITP == 1 && q == 0 && j > 0) {
            if (!rescale) mbar_wait(o_full(t), ofp, 0x680 + t);
            tc_fence_after();
          }
          if (WAITP != 2) tmem_st16(tP + 16 * q, pk[q]);
          if (STAGGER && q == 1 && j == 0 && t == 0 && u.valid[1]) named_bar_arrive(kBarStagger, 256);
        }
        if (WAITP == 2) {
          if (j > 0) {
            if (!rescale) mbar_wait(o_full(t), ofp, 0x680 + t);
            tc_fence_after();
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) tmem_st16(tP + 16 * q, pk[q]);
        }
        if (j > 0) ofp ^= 1u;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float a0, a1;
          f2_unpack(f2_add(f2_add(rs2[h][0], rs2[h][1]), f2_add(rs2[h][2], rs2[h][3])), a0, a1);
          l_sum[h] += a0 + a1;
        }
        stamp(j, 5);
        tmem_st_wait();
        tc_fence_before();
        named_bar_arrive(kBarPF + t, kGroupSync);  // P_t(j) is in tensor memory
        stamp(j, 6);
      };
#pragma unroll 1
      for (int j = 0; j < num_kv - 1; ++j) tile(j, FaTag<false>{});
      if (ragged)
        tile(num_kv - 1, FaTag<true>{});
      else
        tile(num_kv - 1, FaTag<false>{});

      // ---- epilogue: O / l -> bf16 -> swizzled staging tile -> one TMA store per group and unit (rows past N are clipped
      //      by the tensor map). The other group and the tensor pipe keep running.
      mbar_wait(o_full(t), ofp, 0x690 + t);  // the last P V of this unit has retired
      ofp ^= 1u;
      tc_fence_after();
      uint32_t o[2][32];
      tmem_ld32(tO, o[0]);
      tmem_ld32(tO + 32, o[1]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free(t));  // O_t may be overwritten by the next unit's first P V
      const float inv = 1.0f / (l_sum[0] + l_sum[1]);
      if (gthread == 0 && stored) bulk_wait_read<0>();  // the previous unit's store has finished reading the staging tile
      named_bar_sync(kBarWG + t, 128);
      const uint32_t o_row = sO + static_cast<uint32_t>(row) * 128u;
      const uint32_t o_sw = static_cast<uint32_t>(row & 7);
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t chunk = static_cast<uint32_t>(h * 4 + i);
          st_shared_v4(o_row + ((chunk ^ o_sw) << 4),
                       pack_bf16x2(__uint_as_float(o[h][8 * i]) * inv, __uint_as_float(o[h][8 * i + 1]) * inv),
                       pack_bf16x2(__uint_as_float(o[h][8 * i + 2]) * inv, __uint_as_float(o[h][8 * i + 3]) * inv),
                       pack_bf16x2(__uint_as_float(o[h][8 * i + 4]) * inv, __uint_as_float(o[h][8 * i + 5]) * inv),
                       pack_bf16x2(__uint_as_float(o[h][8 * i + 6]) * inv, __uint_as_float(o[h][8 * i + 7]) * inv));
        }
      fence_proxy_async_smem();
      named_bar_sync(kBarWG + t, 128);
      if (gthread == 0) {
        tma_store_3d(&tmap_out, sO, u.head * 64, u.q0 + 128 * t, u.img);
        bulk_commit();
        stored = true;
      }
    }
    if (gthread == 0 && stored) bulk_wait<0>();  // all stores of this group have completed before the CTA retires
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kFaTmemCols);
  }
}

}  // namespace ada
