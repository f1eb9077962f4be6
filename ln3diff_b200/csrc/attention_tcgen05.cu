// Fused multi-head attention forward for sm_100a (head_dim 64, bf16 in, fp32 softmax / accumulate).
//
// Replaces xformers.ops.memory_efficient_attention at its call sites on the path:
//   vit/vision_transformer.py:114-118 (DiT self-attention, (B, N, 3, H, 64) packed qkv),
//   ldm/modules/attention.py:279-307  (cross-attention; the reference's three permute+contiguous
//                                       copies disappear: heads are addressed through the TMA map),
//   dit/dit_decoder.py                (in-plane / global attention of the DiT2 VAE decoder).
// Semantics: out = softmax(q k^T * scale) v (xformers FMHA with attn_bias=None); optionally a causal mask
// (CLIP text tower) or a second K/V source appended after the first (I23D DINO tokens, never concatenated).
//
// Why three softmax warpgroups.  At head_dim 64 the softmax is bound by the XU (MUFU.EX2: 16 lanes/clk/SM, i.e.
// one warp instruction per 8 clocks per scheduler) at twice the tensor time.  An in-kernel timeline of a CTA with two
// softmax warpgroups (profiles/r2_fmha_timeline_self.txt) shows the XU pipe saturated only while BOTH warpgroups are
// inside their exponential loops and idle for about a third of every block period (TMEM load, row maximum, barrier
// round trips), because the two fall into lock-step; a single warp per scheduler cannot keep the pipe busy on its own
// (ptxas batches the MUFUs, an in-order warp then has nothing else to issue).  Here a CTA owns THREE 128-row query
// tiles (one warpgroup each, 12 softmax warps = 3 per scheduler), so while one warpgroup does its bookkeeping the
// other two can keep the XU busy.  KV blocks are 96 rows so that 3 score tiles (3 x 96 fp32 columns) and 3 output
// tiles (3 x 64) fit the 512 TMEM columns; a thread holds 96 scores.  ptxas (CUDA 12.9) reports 128 registers, a
// 72-byte stack frame, 32 bytes of spill stores and 52 bytes of spill loads.
//
// Roles (512 threads): warps 0-11 softmax (warpgroup t = warp / 4 owns query tile t, thread = row = TMEM
// lane), warp 12 TMA producer, warps 13-15 tcgen05.mma issuers (one per tile).
//   TMA : Q (3 tiles, single buffer per item), K ring and V ring (3 stages each, released separately: K of a
//         block is dead two block periods before its V).
//   MMA : S_t(g) = Q_t K(g)^T (128x96x16 x4), O_t += P_t(g) V(g) (128x64x16 x6, V MN-major from the TMA
//         layout).  Issue order per tile: P_t V(g), then Q_t K(g+2)^T as soon as the warpgroup has pulled
//         S_t(g+1) into registers.
// O accumulates in TMEM across KV blocks.  The running maximum is only raised when a block exceeds it by more than
// 2^8 (then the owning thread rescales its O row in TMEM); otherwise P is computed against the stale maximum, which
// is exact after the final 1/l normalisation.  Only the first block of an item pays a separate max pass; later
// blocks track their maximum inside the exponential loop and are redone in the rare case that it passes the
// threshold.
// Work items are (batch, head, 384-query-row) triples dealt round-robin to a persistent grid; the last,
// partial round is dealt as (2 tiles | 1 tile) halves to twice as many SMs when they fit.
#include <type_traits>

#include "common.cuh"
#include "ln3_internal.h"

namespace ln3 {

static constexpr int kQT = 128;    // query rows per tile
static constexpr int kNT = 3;      // query tiles (= softmax warpgroups) per CTA
static constexpr int kKB = 96;     // kv rows per block
static constexpr int kHD = 64;     // head dim
static constexpr int kQBytes = kQT * kHD * 2;    // 16 KB
static constexpr int kKVBytes = kKB * kHD * 2;   // 12 KB
static constexpr int kStages = 3;                // K ring and V ring depth
static constexpr int kPBytes = 2 * kQBytes;      // P_t: two 64-column 128B-swizzle atoms (the second half used)
static constexpr int kSmem = 1024 + kNT * kQBytes + 2 * kStages * kKVBytes + kNT * kPBytes + 512;
static constexpr int kThreads = (4 * kNT + 1 + kNT) * 32;  // 512: 12 softmax warps, TMA warp, 3 MMA warps
static constexpr int kTmemCols = 512;            // S_t at 96 t (t < 3), O_t at 288 + 64 t
static constexpr int kTmemO = kNT * kKB;
static constexpr float kRescaleThreshold = 8.0f;  // log2 units
// Suspend-time hint of every mbarrier wait: a waiting warp sleeps in hardware instead of feeding try_wait / branch
// pairs into the issue slots of the softmax warps it shares a scheduler with (measured against plain polling:
// DESIGN.md section 5c).
static constexpr uint32_t kWaitNs = 2000;

#ifdef LN3_FMHA_TRACE
// Debug timeline (tools/microbench/fmha_trace.cu): CTA 0, first 64 KV blocks; role 0-2 = softmax warpgroups
// (thread 0 of the group), role 3 = MMA.
__device__ long long g_fmha_trace[4][64][12];
#define LN3_TR3(role, blk, slot)                                                   \
  do {                                                                             \
    if (blockIdx.x == 0 && (blk) < 64) g_fmha_trace[role][blk][slot] = clock64();  \
  } while (0)
#else
#define LN3_TR3(role, blk, slot) do {} while (0)
#endif

struct FmhaParams {
  int Lq, Lkv, Lkv2;
  int B, H, nq;          // work items = B * H * nq query-row triples (384 rows each)
  float rcp_nq, rcp_H;
  float scale_log2;
  int full_items, n_split;  // tail schedule: see the file header
  int causal;               // key j visible to query i only when j <= i
};

__global__ void __launch_bounds__(kThreads, 1)
fmha_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_k2,
                const __grid_constant__ CUtensorMap tmap_v2, const __grid_constant__ CUtensorMap tmap_o,
                const FmhaParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                          // [kNT]
  uint8_t* sK = sQ + kNT * kQBytes;            // [kStages]
  uint8_t* sV = sK + kStages * kKVBytes;       // [kStages]
  uint8_t* sP = sV + kStages * kKVBytes;       // [kNT][2 atoms]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + kNT * kPBytes);
  uint64_t* q_full = bars;                     // [1]
  uint64_t* q_empty = bars + 1;                // [1]
  uint64_t* k_full = bars + 2;                 // [kStages]
  uint64_t* k_empty = k_full + kStages;
  uint64_t* v_full = k_empty + kStages;
  uint64_t* v_empty = v_full + kStages;
  uint64_t* s_full = v_empty + kStages;        // [kNT]
  uint64_t* s_empty = s_full + kNT;            // [kNT] 4 arrivals (one per warp): S_t is in registers
  uint64_t* p_full = s_empty + kNT;            // [kNT] 4 arrivals
  uint64_t* o_full = p_full + kNT;             // [kNT]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + kNT);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  constexpr int kTmaWarp = 4 * kNT, kMmaWarp = 4 * kNT + 1;
  const int nkv1 = (p.Lkv + kKB - 1) / kKB;  // a ragged last block of the first source is masked like the final one
  const int nkv = nkv1 + (p.Lkv2 + kKB - 1) / kKB;
  // w = (batch * H + head) * nq + qp; reciprocal multiplies (exact for w < 2^20, checked on the host)
  auto item_coords = [&](int w, int& q0, int& head, int& batch) {
    const int bh = __float2int_rz((static_cast<float>(w) + 0.5f) * p.rcp_nq);
    const int qp = w - bh * p.nq;
    q0 = qp * kNT * kQT;
    batch = __float2int_rz((static_cast<float>(bh) + 0.5f) * p.rcp_H);
    head = bh - batch * p.H;
  };
  // this CTA's schedule: n_full_my round-robin triple items, then (tail schedule) at most one partial item
  const int cta = static_cast<int>(blockIdx.x), ncta = static_cast<int>(gridDim.x);
  const int n_full_my = cta < p.full_items ? (p.full_items - cta + ncta - 1) / ncta : 0;
  const int n_my = n_full_my + (cta < 2 * p.n_split ? 1 : 0);
  // item `it` of this CTA: work item, its coordinates and the set of tiles this CTA computes (0 = nothing)
  auto sched = [&](int it, int& q0, int& head, int& batch) -> int {
    int w, mask;
    if (it < n_full_my) { w = cta + it * ncta; mask = 7; }
    else { w = p.full_items + (cta >> 1); mask = (cta & 1) ? 4 : 3; }
    item_coords(w, q0, head, batch);
    int valid = 0;
#pragma unroll
    for (int t = 0; t < kNT; ++t)
      if (q0 + t * kQT < p.Lq) valid |= 1 << t;
    return mask & valid;
  };

  if (tid == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    tma_prefetch_desc(&tmap_o);
    if (p.Lkv2 > 0) {
      tma_prefetch_desc(&tmap_k2);
      tma_prefetch_desc(&tmap_v2);
    }
    mbar_init(q_full, 1);
    mbar_init(q_empty, kNT);          // one release per MMA warp
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], kNT);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], kNT);
    }
    for (int i = 0; i < kNT; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 4);   // one arrival per softmax warp (elected lane after __syncwarp)
      mbar_init(&p_full[i], 4);
      mbar_init(&o_full[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------ TMA producer
    if ((tid & 31) == 0) {
      int st = 0, ph = 0, n_items = 0;
      for (int it = 0; it < n_my; ++it) {
        int q0, head, batch;
        const int mask = sched(it, q0, head, batch);
        if (mask == 0) continue;
        mbar_wait_hint(q_empty, (n_items & 1) ^ 1, kWaitNs);
        ++n_items;
        mbar_arrive_expect_tx(q_full, __popc(mask) * kQBytes);
        for (int t = 0; t < kNT; ++t)
          if (mask >> t & 1) tma_load_3d(sQ + t * kQBytes, &tmap_q, q_full, head * kHD, q0 + t * kQT, batch);
        for (int j = 0; j < nkv; ++j) {
          const CUtensorMap* mk = j < nkv1 ? &tmap_k : &tmap_k2;
          const CUtensorMap* mv = j < nkv1 ? &tmap_v : &tmap_v2;
          const int r0 = (j < nkv1 ? j : j - nkv1) * kKB;
          mbar_wait_hint(&k_empty[st], ph ^ 1, kWaitNs);
          mbar_arrive_expect_tx(&k_full[st], kKVBytes);
          tma_load_3d(sK + st * kKVBytes, mk, &k_full[st], head * kHD, r0, batch);
          mbar_wait_hint(&v_empty[st], ph ^ 1, kWaitNs);
          mbar_arrive_expect_tx(&v_full[st], kKVBytes);
          tma_load_3d(sV + st * kKVBytes, mv, &v_full[st], head * kHD, r0, batch);
          if (++st == kStages) st = 0, ph ^= 1;
        }
      }
    }
  } else if (warp >= kMmaWarp) {
    // ------------------------------------------------------------ MMA issuers, one warp per query tile
    // A single in-order issuing warp serialises the three tiles: tcgen05.mma issue blocks while the pipe's
    // short queue is full, so every group of 4-6 MMAs costs its execution time plus ~150-300 cycles of wait /
    // fence / commit latency (tools/microbench/umma_rate.cu), and with six groups per KV block P_t sat ~1800
    // cycles in shared memory before its P V was even issued.  With one warp per tile a tile's S -> P -> O chain
    // waits only for its own warpgroup; the three warps' MMAs interleave in the tensor pipe.
    // The whole warp walks this code with warp-uniform values (descriptors stay in uniform registers);
    // elect_one_sync() guards only the tcgen05 instructions.
    const int t = warp - kMmaWarp;
    constexpr uint32_t idesc_s = make_idesc_bf16(128, kKB, 0, 0);
    constexpr uint32_t idesc_o = make_idesc_bf16(128, kHD, 0, 1);  // B (= V) is MN-major
    const uint32_t tm = __shfl_sync(0xffffffffu, tmem_base, 0);
    constexpr uint32_t kQD = kQBytes >> 4, kKVD = kKVBytes >> 4, kPD = kPBytes >> 4;  // descriptor units (16 B)
    const uint64_t dQ = make_smem_desc_sw128(smem_u32(sQ), 0, 1024) + static_cast<uint32_t>(t) * kQD;
    const uint64_t dK = make_smem_desc_sw128(smem_u32(sK), 0, 1024);
    const uint64_t dV = make_smem_desc_sw128(smem_u32(sV), 1024, 1024);
    const uint64_t dP = make_smem_desc_sw128(smem_u32(sP), 0, 1024) + static_cast<uint32_t>(t) * kPD;
    const uint32_t tS = tm + t * kKB, tO = tm + kTmemO + t * kHD;

    // cursor over the (item, block) sequence of this CTA, skipping items with an empty tile set
    struct Cursor { int it, j, mask, st, ph, items; bool end; };
    auto cur_init = [&](Cursor& c) {
      c.it = -1; c.j = nkv - 1; c.mask = 0; c.st = kStages - 1; c.ph = 1; c.items = -1; c.end = false;
    };
    auto cur_next = [&](Cursor& c) {   // advance by one block
      if (++c.st == kStages) c.st = 0, c.ph ^= 1;
      if (++c.j < nkv) return;
      c.j = 0;
      int q0, head, batch;
      do {
        if (++c.it >= n_my) { c.end = true; c.mask = 0; return; }
        c.mask = sched(c.it, q0, head, batch);
      } while (c.mask == 0);
      ++c.items;
    };
    Cursor cq, cp;   // next S block to issue / next P V block to issue
    cur_init(cq);
    cur_init(cp);
    cur_next(cq);
    cur_next(cp);
    int n_qk = 0, n_pv = 0;   // issue counts of this tile (barrier parities)
    int seq = 0;              // trace only

    // S_t of the block under `cq` (or, when the item does not include this tile, only the ring releases)
    auto qk_step = [&]() {
      if (cq.j == 0) mbar_wait_hint(q_full, cq.items & 1, kWaitNs);
      mbar_wait_hint(&k_full[cq.st], cq.ph, kWaitNs);
      if (cq.mask >> t & 1) {
        if (n_qk > 0) mbar_wait_hint(&s_empty[t], (n_qk - 1) & 1, kWaitNs);  // the previous S_t is in registers
        ++n_qk;
        tc_fence_after();
        const uint64_t kd = dK + static_cast<uint32_t>(cq.st) * kKVD;
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < kHD / 16; ++k) umma_f16_ss(tS, dQ + 2 * k, kd + 2 * k, idesc_s, k != 0);
          umma_commit(&s_full[t]);
          umma_commit(&k_empty[cq.st]);
          if (cq.j == nkv - 1) umma_commit(q_empty);
        }
        __syncwarp();
      } else {
        if (elect_one_sync()) {
          mbar_arrive(&k_empty[cq.st]);
          if (cq.j == nkv - 1) mbar_arrive(q_empty);
        }
        __syncwarp();
      }
      LN3_TR3(3, seq, t);
      cur_next(cq);
    };
    auto pv_step = [&]() {
      mbar_wait_hint(&v_full[cp.st], cp.ph, kWaitNs);
      if (cp.mask >> t & 1) {
        const int kv_valid = (cp.j < nkv1) ? p.Lkv - cp.j * kKB : p.Lkv2 - (cp.j - nkv1) * kKB;
        const int ksteps = kv_valid >= kKB ? kKB / 16 : (kv_valid + 15) >> 4;  // P beyond is never written
        const uint64_t vd = dV + static_cast<uint32_t>(cp.st) * kKVD;
        mbar_wait_hint(&p_full[t], n_pv & 1, kWaitNs);  // P_t in smem, O_t rescaled if needed
        ++n_pv;
        LN3_TR3(3, seq, 3 + 2 * t);
        tc_fence_after();
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < kKB / 16; ++k)
            if (k < ksteps)
              umma_f16_ss(tO, dP + (k >> 2) * kQD + (k & 3) * 2, vd + k * 128, idesc_o, (cp.j | k) != 0);
          umma_commit(&o_full[t]);
          umma_commit(&v_empty[cp.st]);
        }
        __syncwarp();
        LN3_TR3(3, seq, 4 + 2 * t);
      } else {
        if (elect_one_sync()) mbar_arrive(&v_empty[cp.st]);
        __syncwarp();
      }
      ++seq;
      cur_next(cp);
    };
    // S(0) and S(1) up front, then per block: P V(g), and S(g+2) as soon as the warpgroup has S(g+1) in registers
    for (int pre = 0; pre < 2 && !cq.end; ++pre) qk_step();
    while (!cp.end) {
      pv_step();
      if (!cq.end) qk_step();
    }
  } else {
    // ------------------------------------------------------------ softmax warpgroups
    const int t = warp >> 2;
    const int row = tid & 127;  // TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tS = tmem_base + t * kKB + lane_off;
    const uint32_t tO = tmem_base + kTmemO + t * kHD + lane_off;
    uint8_t* sPt = sP + t * kPBytes;
    const uint32_t p_row = smem_u32(sPt) + row * 128;
    const int swz = row & 7;
    int g = 0;    // blocks of items this tile took part in (per-tile barrier parities)
    bool o_store_pending = false;  // thread 0 of the group: a bulk store may still be reading P_t's smem
    for (int it = 0; it < n_my; ++it) {
      int q0, head, batch;
      const int mask = sched(it, q0, head, batch);
      if (!(mask >> t & 1)) continue;
      float m_ref = -INFINITY, l_run = 0.f;
      for (int j = 0; j < nkv; ++j, ++g) {
        const int kv_valid = (j < nkv1) ? p.Lkv - j * kKB : p.Lkv2 - (j - nkv1) * kKB;  // >= 1
        if (row == 0) LN3_TR3(t, g, 0);  // start waiting for S
        mbar_wait_hint(&s_full[t], g & 1, kWaitNs);
        if (row == 0) LN3_TR3(t, g, 1);  // S ready
        tc_fence_after();
        uint32_t s[kKB];
        tmem_ld_32x32(tS + 0, s);
        tmem_ld_32x32(tS + 32, s + 32);
        tmem_ld_32x32(tS + 64, s + 64);
        tmem_ld_wait();
        if (row == 0) LN3_TR3(t, g, 2);  // S in registers
        tc_fence_before();
        // one arrival per warp: 128 per-thread arrivals are 128 serialised barrier updates on the MIO queue the
        // exponentials of the other warpgroups are competing for
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&s_empty[t]);  // the tensor core may overwrite S_t with the next block now
        if (kv_valid < kKB) {
#pragma unroll
          for (int i = 0; i < kKB; ++i)
            if (i >= kv_valid) s[i] = 0xff800000u;  // -inf
        }
        if (p.causal) {   // (first K/V source only; every row keeps key 0, so block 0 is never fully masked)
          const int lim = q0 + t * kQT + row - j * kKB;   // columns i > lim are in the future of this row
#pragma unroll
          for (int i = 0; i < kKB; ++i)
            if (i > lim) s[i] = 0xff800000u;
        }
        const int c_end = kv_valid >= kKB ? kKB : (kv_valid + 15) & ~15;  // = 16 * PV k-steps
        // Only the first block of an item pays a separate max pass.  Later blocks exponentiate against the running
        // reference straight away and track their own maximum INSIDE the exponential loop (FMNMX on the ALU pipe, in
        // the issue slots the XU-bound loop leaves free); if the block then turns out to exceed the reference by more
        // than the lazy-rescale threshold -- rare: the threshold is 2^8 -- the block is redone against the new maximum.
        float alpha = 1.f;
        bool need = false;
        if (j == 0) {
          // three independent 3-input max chains
          float mq[3];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            const int b0 = 32 * a;
            mq[a] = fmax3(__uint_as_float(s[b0]), __uint_as_float(s[b0 + 1]), __uint_as_float(s[b0 + 2]));
          }
#pragma unroll
          for (int i = 3; i < 31; i += 2) {
#pragma unroll
            for (int a = 0; a < 3; ++a)
              mq[a] = fmax3(mq[a], __uint_as_float(s[32 * a + i]), __uint_as_float(s[32 * a + i + 1]));
          }
          const float mx = fmax3(fmax3(mq[0], mq[1], mq[2]), __uint_as_float(s[31]),
                                 fmaxf(__uint_as_float(s[63]), __uint_as_float(s[95])));
          m_ref = mx * p.scale_log2;
        }
        if (row == 0) LN3_TR3(t, g, 3);  // max done
        if (j == 0 && g > 0) {  // previous item's O tile left this buffer?  (long done; one barrier per item)
          if (row == 0 && o_store_pending) tma_store_wait_read();
          named_bar_sync(3 + t, kQT);
        }
        // P_t (smem) is read by P_t V of the previous block until o_full fires
        if (g > 0) mbar_wait_hint(&o_full[t], (g - 1) & 1, kWaitNs);
        if (row == 0) LN3_TR3(t, g, 4);  // O of previous block complete
        float rs = 0.f;
        float mb[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // running maxima of this block's scores
        auto exp_store = [&](auto full_tag) {
          constexpr bool FULL = decltype(full_tag)::value;
#pragma unroll
          for (int c = 0; c < kKB; c += 8) {
            if (!FULL && c >= c_end) break;
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              e[i] = fast_exp2(fmaf(__uint_as_float(s[c + i]), p.scale_log2, -m_ref));
              mb[i & 3] = fmaxf(mb[i & 3], __uint_as_float(s[c + i]));
            }
            rs += ((e[0] + e[1]) + (e[2] + e[3])) + ((e[4] + e[5]) + (e[6] + e[7]));
            const uint32_t addr = p_row + (c >> 6) * kQBytes + ((((c & 63) >> 3) ^ swz) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_bf16x2(e[0], e[1])),
                         "r"(pack_bf16x2(e[2], e[3])), "r"(pack_bf16x2(e[4], e[5])),
                         "r"(pack_bf16x2(e[6], e[7]))
                         : "memory");
          }
        };
        if (kv_valid >= kKB) exp_store(std::true_type{});
        else exp_store(std::false_type{});
        if (j > 0) {
          const float m_cand = fmaxf(fmaxf(mb[0], mb[1]), fmaxf(mb[2], mb[3])) * p.scale_log2;
          need = m_cand > m_ref + kRescaleThreshold;
          if (__any_sync(0xffffffffu, need)) {
            // redo the block against the new reference (rows without `need` recompute the same values)
            if (need) {
              alpha = fast_exp2(m_ref - m_cand);
              m_ref = m_cand;
              l_run *= alpha;
            }
            rs = 0.f;
            if (kv_valid >= kKB) exp_store(std::true_type{});
            else exp_store(std::false_type{});
          }
        }
        if (row == 0) LN3_TR3(t, g, 6);  // exponentials done
        l_run += rs;
        if (j > 0 && __any_sync(0xffffffffu, need)) {
          // O_t of the previous block is complete (o_full waited above): rescale it in place
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < kHD; c += 32) {
            uint32_t v[32];
            tmem_ld_32x32(tO + c, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
            tmem_st_32x32(tO + c, v);
          }
          tmem_st_wait();
        }
        fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the tensor core
        tc_fence_before();
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&p_full[t]);
        if (row == 0) LN3_TR3(t, g, 7);  // P handed to the tensor core
      }
      if (row == 0) LN3_TR3(t, g - 1, 8);   // epilogue: start waiting for the last P V
      mbar_wait_hint(&o_full[t], (g - 1) & 1, kWaitNs);
      if (row == 0) LN3_TR3(t, g - 1, 9);   // O complete
      tc_fence_after();
      const float inv = 1.f / l_run;
      // O_t -> bf16 -> this tile's (now idle) P buffer in the 128B-swizzled TMA layout -> one bulk tensor store
#pragma unroll
      for (int c = 0; c < kHD; c += 32) {
        uint32_t v[32];
        tmem_ld_32x32(tO + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          const uint32_t addr = p_row + ((((c + i) >> 3) ^ swz) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr),
                       "r"(pack_bf16x2(__uint_as_float(v[i]) * inv, __uint_as_float(v[i + 1]) * inv)),
                       "r"(pack_bf16x2(__uint_as_float(v[i + 2]) * inv, __uint_as_float(v[i + 3]) * inv)),
                       "r"(pack_bf16x2(__uint_as_float(v[i + 4]) * inv, __uint_as_float(v[i + 5]) * inv)),
                       "r"(pack_bf16x2(__uint_as_float(v[i + 6]) * inv, __uint_as_float(v[i + 7]) * inv))
                       : "memory");
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();  // the TMEM reads above precede the next item's first P_t V (accumulate = 0)
      named_bar_sync(3 + t, kQT);
      if (row == 0) {
        tma_store_3d(sPt, &tmap_o, head * kHD, q0 + t * kQT, batch);
        tma_store_commit();
        o_store_pending = true;
      }
      if (row == 0) LN3_TR3(t, g - 1, 10);  // O stored
    }
    if (row == 0 && o_store_pending) tma_store_wait_all();  // smem must outlive the bulk store
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, kTmemCols);
}

int fmha_fwd(const ln3_fmha_args* a, cudaStream_t stream) {
  if (a->head_dim != kHD) return set_error(LN3_EUNSUPPORTED, "fmha: head_dim must be 64");
  if (a->B <= 0 || a->H <= 0 || a->Lq <= 0 || a->Lkv <= 0)
    return set_error(LN3_EINVAL, "fmha: empty problem");
  if ((a->q_ld | a->k_ld | a->v_ld | a->o_ld | a->q_bs | a->k_bs | a->v_bs | a->o_bs) % 8)
    return set_error(LN3_EINVAL, "fmha: strides must be multiples of 8 elements");
  if ((reinterpret_cast<uintptr_t>(a->q) | reinterpret_cast<uintptr_t>(a->k) |
       reinterpret_cast<uintptr_t>(a->v) | reinterpret_cast<uintptr_t>(a->out)) & 15)
    return set_error(LN3_EINVAL, "fmha: pointers must be 16-byte aligned");
  if (a->causal && (a->k2 != nullptr || a->v2 != nullptr))
    return set_error(LN3_EINVAL, "fmha: causal attention takes a single K/V source");
  if (a->k2 != nullptr || a->v2 != nullptr) {
    if (!a->k2 || !a->v2 || a->Lkv2 <= 0) return set_error(LN3_EINVAL, "fmha: k2/v2/Lkv2 must be given together");
    if ((a->k2_ld | a->v2_ld | a->k2_bs | a->v2_bs) % 8 ||
        ((reinterpret_cast<uintptr_t>(a->k2) | reinterpret_cast<uintptr_t>(a->v2)) & 15))
      return set_error(LN3_EINVAL, "fmha: k2/v2 alignment");
  }
  static DeviceOnce once;   // the shared-memory opt-in is per device
  if (int rc = once.run([] {
        cudaError_t e = cudaFuncSetAttribute(fmha_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        return e == cudaSuccess ? LN3_OK : set_error(LN3_ECUDA, "fmha: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      }))
    return rc;
  const bool two = a->k2 != nullptr;
  CUtensorMap tq, tk, tv, tk2, tv2, to;
  int rc;
  const long long cols = static_cast<long long>(a->H) * kHD;
  if ((rc = make_tmap_3d_bf16(&tq, a->q, cols, a->Lq, a->B, a->q_ld, a->q_bs, kHD, kQT))) return rc;
  if ((rc = make_tmap_3d_bf16(&tk, a->k, cols, a->Lkv, a->B, a->k_ld, a->k_bs, kHD, kKB))) return rc;
  if ((rc = make_tmap_3d_bf16(&tv, a->v, cols, a->Lkv, a->B, a->v_ld, a->v_bs, kHD, kKB))) return rc;
  if ((rc = make_tmap_3d_bf16(&to, a->out, cols, a->Lq, a->B, a->o_ld, a->o_bs, kHD, kQT))) return rc;
  if (two) {
    if ((rc = make_tmap_3d_bf16(&tk2, a->k2, cols, a->Lkv2, a->B, a->k2_ld, a->k2_bs, kHD, kKB))) return rc;
    if ((rc = make_tmap_3d_bf16(&tv2, a->v2, cols, a->Lkv2, a->B, a->v2_ld, a->v2_bs, kHD, kKB))) return rc;
  } else {
    tk2 = tk;
    tv2 = tv;
  }
  FmhaParams p;
  p.Lq = a->Lq;
  p.Lkv = a->Lkv;
  p.Lkv2 = two ? a->Lkv2 : 0;
  p.scale_log2 = a->scale * 1.4426950408889634f;
  p.causal = a->causal ? 1 : 0;
  p.B = a->B;
  p.H = a->H;
  p.nq = (a->Lq + kNT * kQT - 1) / (kNT * kQT);
  p.rcp_nq = 1.0f / static_cast<float>(p.nq);
  p.rcp_H = 1.0f / static_cast<float>(p.H);
  const long long nitems = static_cast<long long>(p.B) * p.H * p.nq;
  if (nitems >= (1 << 20)) return set_error(LN3_EUNSUPPORTED, "fmha: more than 2^20 (batch, head, 384-row) work items");
  const int sms = device_sm_count();
  const int grid = static_cast<int>(nitems < sms ? nitems : sms);
  p.full_items = static_cast<int>(nitems);
  p.n_split = 0;
  // tail schedule: the last, partial round as (2 tiles | 1 tile) halves on twice as many SMs when they fit
  const int rem = static_cast<int>(nitems % grid);
  if (nitems > grid && rem > 0 && 2 * rem <= grid) {
    p.full_items = static_cast<int>(nitems) - rem;
    p.n_split = rem;
  }
  cudaError_t e = launch_pdl(fmha_fwd_kernel, dim3(grid), dim3(kThreads), kSmem, stream, tq, tk, tv, tk2, tv2, to, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(LN3_ECUDA, "fmha launch: %s", cudaGetErrorString(e));
  count_launch();
  return LN3_OK;
}

#ifdef LN3_FMHA_TRACE
int fmha_trace_copy(long long* host) {
  return cudaMemcpyFromSymbol(host, g_fmha_trace, sizeof(g_fmha_trace)) == cudaSuccess ? 0 : 1;
}
#endif

}  // namespace ln3
