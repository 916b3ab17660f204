// Fused ring flash-attention forward for sm_100a.
//
// One persistent, warp-specialised CTA per SM (384 threads):
//   warps 0-3   softmax WG 0   : one thread per query row of Q tile 0 (TMEM lane == row)
//   warps 4-7   softmax WG 1   : same for Q tile 1; the two tiles ping-pong on the tensor core
//   warp 8      TMA producer   : Q tiles and K/V tiles (128B-swizzled tensor-map boxes) -> shared memory
//   warp 9      MMA issuer     : tcgen05.mma  S = Q K^T (SS)  and  O += P V (TS, P in TMEM)
//   warp 10     ring fetcher   : pulls the other ring ranks' K/V slots over NVLink with bulk-TMA copies
//                                (peer global -> smem -> local global) and publishes per-owner ready counters;
//                                also allocates / frees TMEM
//   warp 11     idle (keeps the warpgroup count at three for setmaxnreg)
// (control warps sit on the highest warp ids: the warp scheduler favours them)
//
// TMEM (512 columns): S0 | S1 (128 fp32 columns each, P aliases the first 64 columns as packed 16-bit)
//                     O0 | O1 (D fp32 columns each).  O, the running max and the running sum stay in
// TMEM / registers across every hop of the ring, so nothing is re-normalised or round-tripped through
// HBM between hops (reference: ring_flash_attention_cuda.py:136-186 carries o/m/lse through global
// memory in 16 bit and launches one Triton kernel + one NCCL exchange + barrier per hop).
//
// The ring itself is only a schedule: ring rank r visits owners hop_owner[0..hop_count) (itself first).
// K/V of owner o live in slot o of a symmetric [world][2][b*hk][n][d] buffer.  Slot r is written locally
// by pack_kv; the other slots are filled inside this kernel by the fetcher warps of all CTAs (each moves
// 1/gridDim of every slot), overlapping the NVLink transfer with the MMAs of earlier hops.  Layout
// (plain / striped / zig-zag), causal + sliding-window masking and key padding are position functions
// evaluated in-kernel; fully masked tiles are never loaded.
#include <cstdlib>

#include "attn_common.cuh"

namespace rab {
namespace {

constexpr int BM = 128;
constexpr int BN = 128;
constexpr int NSLOT = 4;
constexpr int FETCH_PIECE = 16384;
constexpr int NTHREADS = 384;
constexpr int SUB_BYTES = 128 * 128;  // one 64-element-wide, 128-row swizzled sub-tile

template <int D>
struct FwdSmem {
  static constexpr int NSUB = D / 64;
  static constexpr int TILE_BYTES = NSUB * SUB_BYTES;
  alignas(1024) uint8_t q[2][TILE_BYTES];
  alignas(1024) uint8_t kv[NSLOT][TILE_BYTES];
  alignas(1024) uint8_t fetch[2][FETCH_PIECE];
  uint64_t q_full[2], q_empty[2];
  uint64_t kv_full[NSLOT], kv_empty[NSLOT];
  uint64_t s_full[2], p_ready[2], o_done[2], epi_done[2];
  uint64_t item_go[2], o_ready[2];  // hop-at-a-time mode: issuer started the item / the carried O sits in TMEM
  uint64_t fetch_full[2];
  uint32_t tmem_base;
};

struct Item {
  int b, h, kvh, qp;
  int row0[2];
  bool tvalid[2];
  int qlo[2], qhi[2];
};

__device__ __forceinline__ int num_items(const AttnFwdParams& p) {
  const int nqp = (p.n_q + 2 * BM - 1) / (2 * BM);
  return p.batch * p.heads * nqp;
}

// Work items are ordered heaviest-first (largest q index first under causal masking) and, inside one
// q-pair, so that query heads sharing a KV head are adjacent (L2 reuse of the K/V tiles).
__device__ __forceinline__ void decode_item(const AttnFwdParams& p, int idx, Item& it) {
  const int bh = p.batch * p.heads;
  const int nqp = (p.n_q + 2 * BM - 1) / (2 * BM);
  it.qp = nqp - 1 - idx / bh;
  const int r = idx % bh;
  it.b = r / p.heads;
  const int hh = r % p.heads;
  const int groups = p.heads / p.kv_heads;
  it.kvh = hh / groups;
  it.h = (hh % groups) * p.kv_heads + it.kvh;  // reference mapping: query head j uses kv head j % kv_heads
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    it.row0[t] = it.qp * 2 * BM + t * BM;
    it.tvalid[t] = it.row0[t] < p.n_q;
    if (it.tvalid[t]) {
      pos_range(p.pos, p.rank, it.row0[t], min(it.row0[t] + BM, p.n_q) - 1, it.qlo[t], it.qhi[t]);
      it.qlo[t] += p.q_pos_offset;
      it.qhi[t] += p.q_pos_offset;
    } else {
      it.qlo[t] = it.qhi[t] = 0;
    }
  }
}

using FwdScan = WarpTileScan<2, false>;

__device__ __forceinline__ void init_scan(FwdScan& sc, const AttnFwdParams& p, const Item& it) {
  sc.pm = &p.pos;
  sc.hop_owner = p.hop_owner;
  sc.hop_count = p.hop_count;
  sc.groups = 1;
  sc.n_stream = p.n_k;
  sc.tile = BN;
  sc.stream_off = 0;
  sc.stat_off = 0;
  sc.mc = MaskCfg{p.causal, p.window, p.kmask_bits != nullptr};
#pragma unroll
  for (int t = 0; t < 2; ++t) sc.st[t] = StatRange{it.qlo[t], it.qhi[t], it.tvalid[t], false};
}

// ------------------------------------------------------------------------------------------------
// warp 0: TMA producer (all 32 lanes scan tiles, lane 0 issues)
// ------------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ void producer_role(FwdSmem<D>& sm, const AttnFwdParams& p, const CUtensorMap* map_q,
                                              const CUtensorMap* map_kv) {
  constexpr int NSUB = FwdSmem<D>::NSUB;
  constexpr uint32_t TILE_BYTES = FwdSmem<D>::TILE_BYTES;
  const int lane = lane_id();
  uint32_t n_slot = 0;
  uint32_t items_t[2] = {0, 0};
  uint32_t ready_mask = p.all_ready ? 0xffffffffu : (1u << p.rank);
  const int total = num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x) {
    Item it;
    decode_item(p, idx, it);
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      if (!it.tvalid[t]) continue;
      if (lane == 0) {
        mbar_wait(&sm.q_empty[t], (items_t[t] & 1) ^ 1, 100 + t);
        mbar_expect_tx(&sm.q_full[t], TILE_BYTES);
#pragma unroll
        for (int s = 0; s < NSUB; ++s)
          tma_load_4d(sm.q[t] + s * SUB_BYTES, map_q, &sm.q_full[t], s * 64, it.h, it.row0[t], it.b);
      }
      items_t[t]++;
    }
    FwdScan scan;
    init_scan(scan, p, it);
    ScanTile ti;
    while (scan.next(lane, ti)) {
      if (!((ready_mask >> ti.owner) & 1u)) {
        if (lane == 0) {
          spin_until_ge_gpu(&p.ready[ti.owner], gridDim.x, 110);
          fence_proxy_async_global();
        }
        ready_mask |= 1u << ti.owner;
      }
      if (lane == 0) {
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          const uint32_t n = n_slot + which;
          const uint32_t slot = n % NSLOT, ph = (n / NSLOT) & 1;
          mbar_wait(&sm.kv_empty[slot], ph ^ 1, 120 + slot);
          mbar_expect_tx(&sm.kv_full[slot], TILE_BYTES);
#pragma unroll
          for (int s = 0; s < NSUB; ++s)
            tma_load_4d(sm.kv[slot] + s * SUB_BYTES, map_kv, &sm.kv_full[slot], s * 64, ti.idx * BN,
                        it.b * p.kv_heads + it.kvh, ti.owner * 2 + which);
        }
      }
      n_slot += 2;
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// warp 1: MMA issuer (all 32 lanes scan tiles, lane 0 issues tcgen05.mma)
// ------------------------------------------------------------------------------------------------
template <int D, bool BF16>
__device__ __forceinline__ void mma_role(FwdSmem<D>& sm, const AttnFwdParams& p, uint32_t tmem_in) {
  constexpr uint32_t idesc_qk = umma_idesc_bf16(BM, BN, 0, 0, BF16 ? 1 : 0);
  constexpr uint32_t idesc_pv = umma_idesc_bf16(BM, D, 0, 1, BF16 ? 1 : 0);
  // K-major operands (Q, K): 8-row groups 1024 B apart; the leading offset is unused with 128B swizzle.
  constexpr uint64_t kmaj_static = umma_smem_desc_hi_lo(16, 1024, UMMA_LAYOUT_SW128);
  // MN-major operand (V as B of P V): 64-wide d sub-tiles SUB_BYTES apart, 8-row kv groups 1024 B apart.
  constexpr uint64_t vmaj_static = umma_smem_desc_hi_lo(SUB_BYTES, 1024, UMMA_LAYOUT_SW128);

  // The whole warp runs this role in lock step with warp-uniform values; the *_w wrappers elect one lane for
  // the actual tcgen05 instruction.  Descriptors are built once and advanced with constant adds.
  const int lane = lane_id();
  const uint32_t tmem = warp_uniform(tmem_in);
  uint32_t n_kv = 0;
  uint32_t cnt_p[2] = {0, 0};
  uint32_t items_t[2] = {0, 0};
  const uint32_t s_tm0 = tmem, s_tm1 = tmem + 128;
  const uint32_t o_tm0 = tmem + 256, o_tm1 = tmem + 256 + D;
  const uint64_t q_desc0 = umma_desc(kmaj_static, smem_u32(sm.q[0]));
  const uint64_t q_desc1 = umma_desc(kmaj_static, smem_u32(sm.q[1]));
  const uint64_t kv_kdesc0 = umma_desc(kmaj_static, smem_u32(sm.kv[0]));
  const uint64_t kv_vdesc0 = umma_desc(vmaj_static, smem_u32(sm.kv[0]));
  constexpr uint32_t SLOT16 = FwdSmem<D>::TILE_BYTES >> 4;

  auto issue_qk = [&](const int t, const uint32_t kslot) {
    const uint64_t kd = kv_kdesc0 + uint64_t(kslot * SLOT16);
    const uint64_t qd = t ? q_desc1 : q_desc0;
    const uint32_t st = t ? s_tm1 : s_tm0;
    if (elect_one()) {  // one election per batch: 8 back-to-back UTCHMMA with 1-3 instructions in between
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk) {
        const uint32_t off = (kk / 4) * SUB_BYTES + (kk % 4) * 32;
        umma_ss(st, umma_desc_add(qd, off), umma_desc_add(kd, off), idesc_qk, kk > 0);
      }
      umma_commit(&sm.s_full[0] + t);
    }
    __syncwarp();
  };

  const int total = num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x) {
    Item it;
    decode_item(p, idx, it);
#pragma unroll
    for (int t = 0; t < 2; ++t)
      if (it.tvalid[t]) mbar_wait(&sm.q_full[t], items_t[t] & 1, 200 + t);
    tc_fence_after();

    const bool carry = p.carry_in != 0;
    if (carry) {
      // the warpgroups may load the carried state of this item now (keeps them in lock step with this warp: they
      // can never run two items ahead, so the parity waits on o_ready stay unambiguous)
#pragma unroll
      for (int t = 0; t < 2; ++t)
        if (it.tvalid[t] && elect_one()) mbar_arrive(&sm.item_go[t]);
      __syncwarp();
    }
    FwdScan scan;
    init_scan(scan, p, it);
    ScanTile cur, nxt;
    bool has = scan.next(lane, cur);
    bool pv_started[2] = {carry, carry};   // a carried O is accumulated into from the first P V on
    bool o_waited[2] = {false, false};
    if (has) {
      const uint32_t ks = (2 * n_kv) % NSLOT, kph = ((2 * n_kv) / NSLOT) & 1;
      mbar_wait(&sm.kv_full[ks], kph, 210);
      tc_fence_after();
#pragma unroll
      for (int t = 0; t < 2; ++t)
        if (cur.need[t]) issue_qk(t, ks);
      umma_commit_w(&sm.kv_empty[ks]);
    }
    while (has) {
      const bool hasn = scan.next(lane, nxt);
      const uint32_t vs = (2 * n_kv + 1) % NSLOT, vph = ((2 * n_kv + 1) / NSLOT) & 1;
      const uint32_t ksn = (2 * n_kv + 2) % NSLOT, kphn = ((2 * n_kv + 2) / NSLOT) & 1;
      mbar_wait(&sm.kv_full[vs], vph, 220);
      tc_fence_after();
      bool kwaited = false;
      const uint64_t vd = kv_vdesc0 + uint64_t(vs * SLOT16);
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        if (cur.need[t]) {
          if (!o_waited[t]) {
            // the O block of this Q tile is ours: the previous item's epilogue has drained it, or (hop mode) the
            // warpgroup has loaded the carried accumulator into it
            if (carry) mbar_wait(&sm.o_ready[t], items_t[t] & 1, 232 + t);
            else mbar_wait(&sm.epi_done[t], (items_t[t] & 1) ^ 1, 230 + t);
            o_waited[t] = true;
          }
          mbar_wait(&sm.p_ready[t], cnt_p[t] & 1, 240 + t);
          tc_fence_after();
          const uint32_t ot = t ? o_tm1 : o_tm0, st = t ? s_tm1 : s_tm0;
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < BN / 16; ++kk) {
              umma_ts(ot, st + kk * 8, umma_desc_add(vd, kk * 2048), idesc_pv, (pv_started[t] || kk > 0) ? 1u : 0u);
            }
            umma_commit(&sm.o_done[t]);
          }
          __syncwarp();
          pv_started[t] = true;
          cnt_p[t]++;
        }
        if (hasn && nxt.need[t]) {
          if (!kwaited) {
            mbar_wait(&sm.kv_full[ksn], kphn, 250);
            tc_fence_after();
            kwaited = true;
          }
          issue_qk(t, ksn);
        }
      }
      umma_commit_w(&sm.kv_empty[vs]);
      if (hasn) umma_commit_w(&sm.kv_empty[ksn]);
      n_kv++;
      cur = nxt;
      has = hasn;
    }
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      if (!it.tvalid[t]) continue;
      if (!o_waited[t]) {
        if (carry) mbar_wait(&sm.o_ready[t], items_t[t] & 1, 262 + t);
        else mbar_wait(&sm.epi_done[t], (items_t[t] & 1) ^ 1, 260 + t);
      }
      umma_commit_w(&sm.q_empty[t]);
      items_t[t]++;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// warp 2: ring fetcher (peer K/V slot -> local slot, 1/gridDim of every slot per CTA)
// ------------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ void fetch_role(FwdSmem<D>& sm, const AttnFwdParams& p) {
  uint32_t fcount = 0;
  const unsigned long long npieces = (p.slot_bytes + FETCH_PIECE - 1) / FETCH_PIECE;
  const unsigned long long t_begin = global_timer_ns();
  for (int s = 1; s < p.hop_count; ++s) {
    const int o = p.hop_owner[s];
    const uint8_t* src = p.kv_peer[o];  // owner o's own slot (peer-mapped staging)
    uint8_t* dst = p.kv_local + (unsigned long long)o * p.slot_bytes;
    auto piece_bytes = [&](unsigned long long pc) -> uint32_t {
      const unsigned long long rem = p.slot_bytes - pc * FETCH_PIECE;
      return rem < (unsigned long long)FETCH_PIECE ? (uint32_t)rem : (uint32_t)FETCH_PIECE;
    };
    unsigned long long pc = blockIdx.x;
    if (pc < npieces) {
      // software pipeline: load(i+1) is in flight while load(i) is drained to local memory
      bulk_wait_read<0>();
      {
        const uint32_t buf = fcount & 1;
        const uint32_t bytes = piece_bytes(pc);
        mbar_expect_tx(&sm.fetch_full[buf], bytes);
        bulk_load_1d(sm.fetch[buf], src + pc * FETCH_PIECE, bytes, &sm.fetch_full[buf]);
      }
      while (pc < npieces) {
        const unsigned long long pn = pc + gridDim.x;
        if (pn < npieces) {
          bulk_wait_read<0>();  // the store that last read the other buffer has drained it
          const uint32_t buf = (fcount + 1) & 1;
          const uint32_t bytes = piece_bytes(pn);
          mbar_expect_tx(&sm.fetch_full[buf], bytes);
          bulk_load_1d(sm.fetch[buf], src + pn * FETCH_PIECE, bytes, &sm.fetch_full[buf]);
        }
        const uint32_t buf = fcount & 1;
        mbar_wait(&sm.fetch_full[buf], (fcount >> 1) & 1, 300 + buf);
        bulk_store_1d(dst + pc * FETCH_PIECE, sm.fetch[buf], piece_bytes(pc));
        bulk_commit();
        fcount++;
        pc = pn;
      }
      bulk_wait<0>();  // all stores of this owner's slot are complete
    }
    fence_proxy_async_global();
    __threadfence();
    red_release_gpu_add(&p.ready[o], 1u);
  }
  if (p.fetch_times != nullptr && p.hop_count > 1) {  // bench.py: ring K/V GB/s over the fetch-active window
    p.fetch_times[2 * blockIdx.x] = t_begin;
    p.fetch_times[2 * blockIdx.x + 1] = global_timer_ns();
  }
}

// ------------------------------------------------------------------------------------------------
// warps 4-11: softmax / correction / epilogue, one thread per query row
//
// The 128 logits of a row are consumed as four 32-column chunks in a rolled loop (two chunks per iteration,
// ping-pong registers): the tcgen05.ld of chunk c+1 is in flight while chunk c runs through exp2, and the
// loop body stays small enough for the instruction cache (the fully unrolled 128-wide version spent a quarter
// of its samples in no_instructions stalls, profiles/ncu_r1a_*).  This is an online softmax at chunk
// granularity with a *lazy* running maximum: the maximum is only raised when a chunk exceeds it by more than
// 2^8, in which case l, O (TMEM) and the P chunks of the current tile already written are rescaled.
// ------------------------------------------------------------------------------------------------
template <bool BF16>
__device__ __forceinline__ uint32_t scale_packed(uint32_t w, float f) {
  float a, b;
  if (BF16) {
    a = __uint_as_float(w << 16);
    b = __uint_as_float(w & 0xffff0000u);
    return pack_bf16x2(a * f, b * f);
  } else {
    const __half2 h = *reinterpret_cast<const __half2*>(&w);
    a = __low2float(h);
    b = __high2float(h);
    return pack_f16x2(a * f, b * f);
  }
}

// POLYQ of every 4 logit pairs take their exponential on the FMA pipe (poly_exp2x2) instead of the MUFU.  Measured on
// a B200 at n=65536, h=8, causal with none / a quarter / half of them there: 926 / 976 / 957 TFLOP/s (the MUFU phase of
// a softmax warp shrinks; at one half the extra FMA-pipe instructions start to cost more than the MUFU time they save).
constexpr int POLYQ = 1;

template <int D, bool BF16>
__device__ __forceinline__ void softmax_role(FwdSmem<D>& sm, const AttnFwdParams& p, const int t, uint32_t tmem) {
  const int wg_tid = threadIdx.x - 128 * t;
  const uint32_t lane_off = uint32_t((wg_tid / 32) * 32) << 16;
  const uint32_t s_tm = tmem + t * 128 + lane_off;
  const uint32_t o_tm = tmem + 256 + t * D + lane_off;
  const int lane = lane_id();
  uint64_t* const s_full = &sm.s_full[0] + t;
  uint64_t* const p_ready = &sm.p_ready[0] + t;
  uint64_t* const o_done = &sm.o_done[0] + t;
  uint64_t* const epi_done = &sm.epi_done[0] + t;
  uint32_t cnt = 0;
  uint32_t n_items = 0;  // valid items of this warpgroup so far (hop mode barriers)

  const bool clamp = p.softclamp > 0.f;
  const float mul = clamp ? 1.f : p.scale * kLog2e;
  const float pre = clamp ? p.scale / p.softclamp : 0.f;
  const float post = clamp ? p.softclamp * kLog2e : 0.f;

  const int total = num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x) {
    Item it;
    decode_item(p, idx, it);
    const bool tvalid = t ? it.tvalid[1] : it.tvalid[0];
    if (!tvalid) continue;
    const int row0 = t ? it.row0[1] : it.row0[0];
    const int grow = row0 + wg_tid;
    const bool row_ok = grow < p.n_q;
    const int pos_q = pos_of(p.pos, p.rank, min(grow, p.n_q - 1)) + p.q_pos_offset;

    float m_used = -INFINITY;
    float l = 0.f;
    bool have_o = false;
    uint32_t cnt_item = 0;
    if (p.carry_in) {
      // hop-at-a-time mode: O / m / l of this row continue from the previous hop's launch.  The O block is free (this
      // thread drained it in the previous item's epilogue); the issuer waits on o_ready before its first P V.
      mbar_wait(&sm.item_go[t], n_items & 1, 430 + t);
      const size_t mlrow = ((size_t)it.b * p.heads + it.h) * p.n_q + (row_ok ? grow : 0);
      m_used = row_ok ? p.carry_ml[mlrow] : -INFINITY;
      l = row_ok ? p.carry_ml[(size_t)p.batch * p.heads * p.n_q + mlrow] : 0.f;
      const float4* crow = reinterpret_cast<const float4*>(
          p.carry_o + (((size_t)it.b * p.n_q + (row_ok ? grow : 0)) * p.heads + it.h) * D);
#pragma unroll 1
      for (int c = 0; c < D; c += 32) {
        uint32_t orr[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 x = row_ok ? crow[c / 4 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
          orr[4 * i + 0] = __float_as_uint(x.x);
          orr[4 * i + 1] = __float_as_uint(x.y);
          orr[4 * i + 2] = __float_as_uint(x.z);
          orr[4 * i + 3] = __float_as_uint(x.w);
        }
        tmem_st32(o_tm + c, orr);
      }
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(&sm.o_ready[t]);
      have_o = true;
    }
    n_items++;

    FwdScan scan;
    init_scan(scan, p, it);
    ScanTile ti;
    while (scan.next(lane, ti)) {
      const bool need = t ? ti.need[1] : ti.need[0];
      if (!need) continue;
      const bool part = t ? ti.part[1] : ti.part[0];
      mbar_wait(s_full, cnt & 1, 400 + t);
      tc_fence_after();

      // per-tile mask context (only used on partial tiles)
      const int c0 = ti.idx * BN;
      const int split = p.pos.seg_len - c0;
      const int a0 = p.pos.base0[ti.owner] + p.pos.stride * c0;
      const int a1 = p.pos.base1[ti.owner] + p.pos.stride * (c0 - p.pos.seg_len);
      const int ncols = p.n_k - c0;
      uint32_t mb0 = 0xffffffffu, mb1 = 0xffffffffu, mb2 = 0xffffffffu, mb3 = 0xffffffffu;
      if (part && p.kmask_bits != nullptr) {
        const uint32_t* w = p.kmask_bits + ((size_t)ti.owner * p.batch + it.b) * p.kmask_words + (size_t)ti.idx * 4;
        mb0 = w[0]; mb1 = w[1]; mb2 = w[2]; mb3 = w[3];
      }

      float2 ls01 = make_float2(0.f, 0.f), ls23 = make_float2(0.f, 0.f);

      // one 32-column chunk: mask, lazy max, exp2, pack, store P chunk
      auto process = [&](uint32_t (&x)[32], const int c) {
        if (clamp) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = __float_as_uint(fast_tanh(__uint_as_float(x[j]) * pre) * post);
        }
        if (part) {
          const uint32_t mbits = c == 0 ? mb0 : (c == 1 ? mb1 : (c == 2 ? mb2 : mb3));
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            const int pk = (col < split ? a0 : a1) + p.pos.stride * col;
            bool keep = (col < ncols) && ((mbits >> j) & 1u);
            if (p.causal) {
              keep = keep && (pk <= pos_q);
              if (p.window > 0) keep = keep && (pos_q - pk <= p.window);
            }
            if (!keep) x[j] = 0xff800000u;  // -inf
          }
        }
        float m0 = fmaxf(__uint_as_float(x[0]), __uint_as_float(x[1]));
        float m1 = fmaxf(__uint_as_float(x[2]), __uint_as_float(x[3]));
#pragma unroll
        for (int j = 4; j < 32; j += 4) {
          m0 = fmaxf(m0, fmaxf(__uint_as_float(x[j]), __uint_as_float(x[j + 1])));
          m1 = fmaxf(m1, fmaxf(__uint_as_float(x[j + 2]), __uint_as_float(x[j + 3])));
        }
        const float cmax = fmaxf(m0, m1) * mul;
        if (__any_sync(0xffffffffu, cmax > m_used + 8.f)) {
          // raise the running max (rare): rescale l, O and the P chunks of this tile written so far
          const float m_new = fmaxf(m_used, cmax);
          const float factor = (m_used == -INFINITY) ? 0.f : fast_exp2(m_used - m_new);
          l *= factor;
          ls01 = fmul2(ls01, make_float2(factor, factor));
          ls23 = fmul2(ls23, make_float2(factor, factor));
          if (have_o) {
            // the previous P V of this Q tile completed before S became visible (commit ordering)
#pragma unroll 1
            for (int cc = 0; cc < D; cc += 32) {
              uint32_t orr[32];
              tmem_ld32(o_tm + cc, orr);
              tc_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; ++i) orr[i] = __float_as_uint(__uint_as_float(orr[i]) * factor);
              tmem_st32(o_tm + cc, orr);
            }
          }
#pragma unroll 1
          for (int cc = 0; cc < c; ++cc) {
            const uint32_t pcol = cc * 16;
            uint32_t pw[16];
            tmem_ld16(s_tm + pcol, pw);
            tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) pw[i] = scale_packed<BF16>(pw[i], factor);
            tmem_st16(s_tm + pcol, pw);
          }
          m_used = m_new;
        }
        const float m_eff = (m_used == -INFINITY) ? 0.f : m_used;
        const float2 mul2 = make_float2(mul, mul), negm2 = make_float2(-m_eff, -m_eff);
        uint32_t w16[16];
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          // packed FFMA2 / FADD2: two logits per issue slot
          const float2 a = ffma2(make_float2(__uint_as_float(x[2 * i]), __uint_as_float(x[2 * i + 1])), mul2, negm2);
          const float2 bq = ffma2(make_float2(__uint_as_float(x[2 * i + 2]), __uint_as_float(x[2 * i + 3])), mul2, negm2);
          // pair index inside the chunk: i (pa), i + 1 (pb)
          const float2 pa = ((i & 3) < POLYQ) ? poly_exp2x2(a) : make_float2(fast_exp2(a.x), fast_exp2(a.y));
          const float2 pb = (((i + 1) & 3) < POLYQ) ? poly_exp2x2(bq) : make_float2(fast_exp2(bq.x), fast_exp2(bq.y));
          ls01 = fadd2(ls01, pa);
          ls23 = fadd2(ls23, pb);
          w16[i] = BF16 ? pack_bf16x2(pa.x, pa.y) : pack_f16x2(pa.x, pa.y);
          w16[i + 1] = BF16 ? pack_bf16x2(pb.x, pb.y) : pack_f16x2(pb.x, pb.y);
        }
        tmem_st16(s_tm + c * 16, w16);
      };

      uint32_t xa[32], xb[32];
      {
        tmem_ld32(s_tm, xa);
#pragma unroll 1
        for (int c = 0; c < 4; c += 2) {
          tc_wait_ld();                      // chunk c has landed
          tmem_ld32(s_tm + (c + 1) * 32, xb);  // chunk c+1 in flight during the math of chunk c
          process(xa, c);
          tc_wait_ld();                      // chunk c+1 has landed
          if (c + 2 < 4) tmem_ld32(s_tm + (c + 2) * 32, xa);
          process(xb, c + 1);
        }
      }
      l += (ls01.x + ls01.y) + (ls23.x + ls23.y);
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(p_ready);
      cnt++;
      cnt_item++;
      have_o = true;
    }

    // epilogue: O / l -> 16 bit, lse
    if (cnt_item > 0) {
      mbar_wait(o_done, (cnt - 1) & 1, 410 + t);
      tc_fence_after();
    }
    if (p.carry_out) {
      // hand the un-normalised state to the next hop's launch
      float4* crow = reinterpret_cast<float4*>(p.carry_o + (((size_t)it.b * p.n_q + (row_ok ? grow : 0)) * p.heads + it.h) * D);
#pragma unroll 1
      for (int c = 0; c < D; c += 32) {
        uint32_t orr[32];
        if (cnt_item > 0 || p.carry_in) {
          tmem_ld32(o_tm + c, orr);
          tc_wait_ld();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) orr[i] = 0u;
        }
        if (row_ok) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            crow[c / 4 + i] = make_float4(__uint_as_float(orr[4 * i]), __uint_as_float(orr[4 * i + 1]),
                                          __uint_as_float(orr[4 * i + 2]), __uint_as_float(orr[4 * i + 3]));
        }
      }
      if (row_ok) {
        const size_t mlrow = ((size_t)it.b * p.heads + it.h) * p.n_q + grow;
        p.carry_ml[mlrow] = m_used;
        p.carry_ml[(size_t)p.batch * p.heads * p.n_q + mlrow] = l;
      }
      tc_fence_before();
      mbar_arrive(epi_done);
      continue;
    }
    const float inv = l > 0.f ? 1.f / l : 0.f;
    uint4* orow = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.o) +
                                           (((size_t)it.b * p.n_q + (row_ok ? grow : 0)) * p.heads + it.h) * D);
#pragma unroll 1
    for (int c = 0; c < D; c += 32) {
      uint32_t orr[32];
      if (cnt_item > 0 || p.carry_in) {
        tmem_ld32(o_tm + c, orr);
        tc_wait_ld();
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) orr[i] = 0u;
      }
      uint32_t w[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float a = __uint_as_float(orr[2 * i]) * inv, bq = __uint_as_float(orr[2 * i + 1]) * inv;
        w[i] = BF16 ? pack_bf16x2(a, bq) : pack_f16x2(a, bq);
      }
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 4; ++i) orow[c / 8 + i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
      }
    }
    if (row_ok) {
      const float m_eff = (m_used == -INFINITY) ? 0.f : m_used;
      p.lse[((size_t)it.b * p.heads + it.h) * p.n_q + grow] = l > 0.f ? (m_eff + log2f(l)) * kLn2 : INFINITY;
    }
    tc_fence_before();
    mbar_arrive(epi_done);
  }
}

template <int D, bool BF16>
__global__ void __launch_bounds__(NTHREADS, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                const __grid_constant__ AttnFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  FwdSmem<D>& sm =
      *reinterpret_cast<FwdSmem<D>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x / 32;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.q_full[i], 1);
      mbar_init(&sm.q_empty[i], 1);
      mbar_init(&sm.s_full[i], 1);
      mbar_init(&sm.p_ready[i], 128);
      mbar_init(&sm.o_done[i], 1);
      mbar_init(&sm.epi_done[i], 128);
      mbar_init(&sm.fetch_full[i], 1);
      mbar_init(&sm.item_go[i], 1);
      mbar_init(&sm.o_ready[i], 128);
    }
    for (int i = 0; i < NSLOT; ++i) {
      mbar_init(&sm.kv_full[i], 1);
      mbar_init(&sm.kv_empty[i], 1);
    }
    fence_mbar_init();
  }
  // warps 0-7: softmax warpgroups (TMEM lane quadrant = warp % 4); warps 8-11: producer, MMA issuer, fetcher.
  // The warp scheduler favours higher warp ids, so the latency-critical issuing warps sit on top.
  if (warp == 8 && lane_id() == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_kv);
  }
  if (warp == 10) {
    tmem_alloc(&sm.tmem_base, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  if (warp >= 8) {
    setmaxnreg_dec<120>();
    if (warp == 8) {
      producer_role<D>(sm, p, &map_q, &map_kv);
    } else if (warp == 9) {
      mma_role<D, BF16>(sm, p, tmem);
    } else if (warp == 10) {
      if (lane_id() == 0) fetch_role<D>(sm, p);
    }
  } else {
    setmaxnreg_inc<192>();
    softmax_role<D, BF16>(sm, p, warp < 4 ? 0 : 1, tmem);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 10) tmem_dealloc(tmem, 512);
}

}  // namespace

size_t attn_fwd_smem_bytes(int head_dim) {
  return (head_dim == 128 ? sizeof(FwdSmem<128>) : sizeof(FwdSmem<64>)) + 1024;
}

template <int D>
void launch_attn_fwd(const CUtensorMap& map_q, const CUtensorMap& map_kv, const AttnFwdParams& p, int num_sms,
                     cudaStream_t stream) {
  using Kern = void (*)(const CUtensorMap, const CUtensorMap, const AttnFwdParams);
  const Kern kern = p.is_bf16 ? attn_fwd_kernel<D, true> : attn_fwd_kernel<D, false>;
  const size_t smem = sizeof(FwdSmem<D>) + 1024;
  cuda_check(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
             "attn_fwd smem attribute");
  const int nqp = (p.n_q + 2 * BM - 1) / (2 * BM);
  const int items = p.batch * p.heads * nqp;
  void* args[] = {(void*)&map_q, (void*)&map_kv, (void*)&p};
  if (p.hop_count > 1) {
    // every CTA owns a share of the NVLink fetch and other CTAs spin on it: all CTAs must be co-resident
    cuda_check(cudaLaunchCooperativeKernel((void*)kern, dim3(num_sms), dim3(NTHREADS), args, smem, stream),
               "attn_fwd cooperative launch");
  } else {
    const int grid = items < num_sms ? items : num_sms;
    cuda_check(cudaLaunchKernel((void*)kern, dim3(grid), dim3(NTHREADS), args, smem, stream), "attn_fwd launch");
  }
}

template void launch_attn_fwd<64>(const CUtensorMap&, const CUtensorMap&, const AttnFwdParams&, int, cudaStream_t);
template void launch_attn_fwd<128>(const CUtensorMap&, const CUtensorMap&, const AttnFwdParams&, int, cudaStream_t);

}  // namespace rab
