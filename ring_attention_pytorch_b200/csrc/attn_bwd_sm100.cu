// Fused ring flash-attention backward for sm_100a: two warp-specialised tcgen05 kernels.
//
//   attn_bwd_dq_kernel   (Q-stationary)  per 128-row query tile, for every visible K/V tile:
//        S = Q K^T (SS) -> P = exp2(S*c - lse)          dP = dO V^T (SS)
//        dS = P o (dP - delta) * scale -> 16 bit in TMEM   dQ += dS K (TS, K as MN-major B)
//   attn_bwd_dkdv_kernel (KV-stationary) per 128-key tile, for every query tile (64 rows) that can see it:
//        S^T = K Q^T, dP^T = V dO^T (SS)                 P^T, dS^T -> 16 bit in TMEM
//        dV += P^T dO, dK += dS^T Q (TS, dO / Q as MN-major B)
//
// Accumulators (dQ, or dK and dV) stay in TMEM for the whole ring: every rank finishes its own dQ, dK
// and dV locally, so the backward needs neither atomics nor a cross-rank reduction.  The price is 7
// instead of 5 GEMMs per tile pair; the reference (ring_flash_attention_cuda.py:211-351) runs a 5-GEMM
// Triton kernel per hop but ships K, V, dK, dV around the ring in 16 bit, adds one extra dK/dV hop per
// iteration and accumulates dQ through global read-modify-write.
//
// Both kernels run two independent "streams" (even / odd streamed tiles), each owning TMEM blocks and a 128-thread
// warpgroup, and two MMA-issuing warps whose waits are blocking in-order mbarrier waits.
//
// This pair is the backward of head dim 64 and the deterministic alternative at head dim 128, where the default is
// the one-kernel, 5-GEMM backward in attn_bwd_fused_sm100.cu.
//
// Inputs are the *gathered* ring buffers (see kernels.h); remote slots are published through ready flags.  In hop mode
// (memory = "ring", one launch per ring hop) the softmax warpgroups load each item's accumulator rows from the fp32
// carry into TMEM before the first accumulating MMA and the epilogue stores them back: the launches perform the same
// fp32 operations in the same order as one launch over every hop.
#include "attn_common.cuh"

namespace rab {
namespace {

constexpr int NTHREADS = 384;
constexpr int SUB128 = 128 * 128;  // 64-element-wide sub-tile, 128 rows
constexpr int SUB64 = 64 * 128;    // 64-element-wide sub-tile, 64 rows

__device__ __forceinline__ void wait_owner_ready(const AttnBwdParams& p, int owner, uint32_t& mask, int tag) {
  if ((mask >> owner) & 1u) return;
  if (p.ready != nullptr) {
    spin_until_ge_gpu(p.ready + owner, p.ready_target, tag);
    fence_proxy_async_global();
  }
  mask |= 1u << owner;
}

// =================================================================================================
// dQ kernel
// =================================================================================================
template <int D>
struct DqSmem {
  static constexpr int NSUB = D / 64;
  static constexpr int TILE = NSUB * SUB128;
  alignas(1024) uint8_t q[TILE];
  alignas(1024) uint8_t dout[TILE];
  alignas(1024) uint8_t k[3][TILE];
  alignas(1024) uint8_t v[2][TILE];
  uint64_t qdo_full, qdo_empty;
  uint64_t k_full[3], k_empty[3];
  uint64_t v_full[2], v_empty[2];
  uint64_t r_s_full[3], r_s_taken[3], r_dp_full[3], r_ds_ready[3], r_free[3];  // per TMEM region
  uint64_t dq_done, epi_done;
  uint64_t carry_ready;  // hop mode: both warpgroups have loaded the item's carried dQ into TMEM
  uint32_t tmem_base;
};

// Before an item's first accumulating MMA the accumulating issuer waits until the accumulator block is its own: the
// previous item's epilogue has drained it, or (hop mode) the warpgroups have loaded the carried accumulator into it,
// which they do only after that epilogue.  Either barrier completes once per item, and the warpgroups arrive for item
// i + 1 only after the issuer's commit of item i, which follows this wait: neither can run two phases ahead.
__device__ __forceinline__ void wait_acc_free(const AttnBwdParams& p, uint64_t* epi_done, uint64_t* carry_ready,
                                              uint32_t n_item, int tag) {
  if (p.carry_in) mbar_wait(carry_ready, n_item & 1, tag + 1);
  else mbar_wait(epi_done, (n_item & 1) ^ 1, tag);
}

// hop mode: one thread's row of its warpgroup's accumulator columns, fp32 carry -> TMEM (zeros for rows past the end)
template <int NCOL>
__device__ __forceinline__ void carry_load(const float* src, bool row_ok, uint32_t taddr) {
  const float4* crow = reinterpret_cast<const float4*>(src);
#pragma unroll 1
  for (int c = 0; c < NCOL; c += 32) {
    uint32_t v[32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 x = row_ok ? crow[c / 4 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
      v[4 * i + 0] = __float_as_uint(x.x);
      v[4 * i + 1] = __float_as_uint(x.y);
      v[4 * i + 2] = __float_as_uint(x.z);
      v[4 * i + 3] = __float_as_uint(x.w);
    }
    tmem_st32(taddr + c, v);
  }
  tc_wait_st();
}

// hop mode: TMEM -> fp32 carry (zeros when the accumulator was never written)
template <int NCOL>
__device__ __forceinline__ void carry_store(float* dst, bool row_ok, bool any, uint32_t taddr) {
  float4* crow = reinterpret_cast<float4*>(dst);
#pragma unroll 1
  for (int c = 0; c < NCOL; c += 32) {
    uint32_t v[32];
    if (any) {
      tmem_ld32(taddr + c, v);
      tc_wait_ld();
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = 0u;
    }
    if (row_ok) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        crow[c / 4 + i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                      __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
    }
  }
}

struct DqItem {
  int b, h, kvh, qt, row0;
  int qlo, qhi;
};

__device__ __forceinline__ int dq_num_items(const AttnBwdParams& p) {
  return p.batch * p.heads * ((p.n_q + 127) / 128);
}

__device__ __forceinline__ void dq_decode(const AttnBwdParams& p, int idx, DqItem& it) {
  const int bh = p.batch * p.heads;
  const int nqt = (p.n_q + 127) / 128;
  it.qt = nqt - 1 - idx / bh;
  const int r = idx % bh;
  it.b = r / p.heads;
  const int hh = r % p.heads;
  const int groups = p.heads / p.kv_heads;
  it.kvh = hh / groups;
  it.h = (hh % groups) * p.kv_heads + it.kvh;
  it.row0 = it.qt * 128;
  pos_range(p.pos, p.rank, it.row0, min(it.row0 + 128, p.n_q) - 1, it.qlo, it.qhi);
  it.qlo += p.q_pos_offset;
  it.qhi += p.q_pos_offset;
}

using DqScan = WarpTileScan<1, false>;

__device__ __forceinline__ void dq_init_scan(DqScan& sc, const AttnBwdParams& p, const DqItem& it) {
  sc.pm = &p.pos;
  sc.hop_owner = p.hop_owner;
  sc.hop_count = p.hop_count;
  sc.groups = 1;
  sc.n_stream = p.n_k;
  sc.tile = 128;
  sc.stream_off = 0;
  sc.stat_off = 0;
  sc.mc = MaskCfg{p.causal, p.window, p.kmask_bits != nullptr};
  sc.st[0] = StatRange{it.qlo, it.qhi, true, false};
}

template <int D>
__device__ __forceinline__ void dq_producer(DqSmem<D>& sm, const AttnBwdParams& p, const CUtensorMap* map_qd,
                                            const CUtensorMap* map_kv) {
  constexpr int NSUB = DqSmem<D>::NSUB;
  constexpr uint32_t TILE = DqSmem<D>::TILE;
  const int lane = lane_id();
  uint32_t n_item = 0, n_tile = 0;
  uint32_t ready_mask = 1u << p.rank;
  const int total = dq_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DqItem it;
    dq_decode(p, idx, it);
    if (lane == 0) {
      mbar_wait(&sm.qdo_empty, (n_item & 1) ^ 1, 500);
      mbar_expect_tx(&sm.qdo_full, 2 * TILE);
#pragma unroll
      for (int s = 0; s < NSUB; ++s) {
        tma_load_4d(sm.q + s * SUB128, map_qd, &sm.qdo_full, s * 64, it.row0, it.b * p.heads + it.h, p.rank * 2);
        tma_load_4d(sm.dout + s * SUB128, map_qd, &sm.qdo_full, s * 64, it.row0, it.b * p.heads + it.h,
                    p.rank * 2 + 1);
      }
    }
    DqScan scan;
    dq_init_scan(scan, p, it);
    ScanTile t;
    while (scan.next(lane, t)) {
      if (lane == 0) {
        wait_owner_ready(p, t.owner, ready_mask, 501);
        const uint32_t ks = n_tile % 3, kph = (n_tile / 3) & 1;
        mbar_wait(&sm.k_empty[ks], kph ^ 1, 510 + ks);
        mbar_expect_tx(&sm.k_full[ks], TILE);
#pragma unroll
        for (int s = 0; s < NSUB; ++s)
          tma_load_4d(sm.k[ks] + s * SUB128, map_kv, &sm.k_full[ks], s * 64, t.idx * 128,
                      it.b * p.kv_heads + it.kvh, t.owner * 2);
        const uint32_t vs = n_tile % 2, vph = (n_tile / 2) & 1;
        mbar_wait(&sm.v_empty[vs], vph ^ 1, 520 + vs);
        mbar_expect_tx(&sm.v_full[vs], TILE);
#pragma unroll
        for (int s = 0; s < NSUB; ++s)
          tma_load_4d(sm.v[vs] + s * SUB128, map_kv, &sm.v_full[vs], s * 64, t.idx * 128,
                      it.b * p.kv_heads + it.kvh, t.owner * 2 + 1);
      }
      n_tile++;
      __syncwarp();
    }
  }
}

// Two issuing warps (same reasoning as dkv_issue_s below: a single issuing warp's polling loop, not the tensor pipe,
// paced the first version of this kernel).  The logits live in three rotating TMEM regions (tile g of this CTA's lifetime
// uses region g % 3, which is also its K smem stage), every barrier between the issuers and the warpgroups is indexed
// by region with parity (g / 3) & 1, and all waits are blocking waits in program order:
//   warp 9  : S(j) = Q K^T into region r, dP(j) = dO V^T into region r once the warpgroup holds S(j) in registers
//   warp 10 : dQ += dS(j) K with dS read from region r; frees the region and the K stage
// A region is reused only after the dQ MMA that read it has completed, so no barrier can run two phases ahead.
__device__ __forceinline__ uint32_t dq_region_col(uint32_t r) { return r == 0 ? 0u : (r == 1 ? 128u : 384u); }

template <int D, bool BF16>
__device__ __forceinline__ void dq_issue_sdp(DqSmem<D>& sm, const AttnBwdParams& p, uint32_t tmem_in) {
  constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, 0, 0, BF16 ? 1 : 0);
  constexpr uint64_t kmaj = umma_smem_desc_hi_lo(16, 1024, UMMA_LAYOUT_SW128);
  constexpr uint32_t SLOT16 = DqSmem<D>::TILE >> 4;
  const int lane = lane_id();
  const uint32_t tmem = warp_uniform(tmem_in);
  uint32_t n_item = 0, tile_base = 0;
  const int total = dq_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DqItem it;
    dq_decode(p, idx, it);
    DqScan scan;
    dq_init_scan(scan, p, it);
    const uint32_t ntiles = scan.count(lane);
    mbar_wait(&sm.qdo_full, n_item & 1, 600);
    tc_fence_after();
    const uint64_t q_desc = umma_desc(kmaj, smem_u32(sm.q)), do_desc = umma_desc(kmaj, smem_u32(sm.dout));
    const uint64_t k_kdesc0 = umma_desc(kmaj, smem_u32(sm.k[0])), v_kdesc0 = umma_desc(kmaj, smem_u32(sm.v[0]));

    auto issue_s = [&](uint32_t j) {
      const uint32_t g = tile_base + j;
      const uint32_t r = g % 3, ph = (g / 3) & 1;
      mbar_wait(&sm.k_full[r], ph, 620 + r);
      if (g >= 3) mbar_wait(&sm.r_free[r], ph ^ 1, 630 + r);  // previous use of the region has been drained by dQ
      tc_fence_after();
      const uint32_t x_tm = tmem + dq_region_col(r);
      const uint64_t kd = k_kdesc0 + uint64_t(r * SLOT16);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t off = (kk / 4) * SUB128 + (kk % 4) * 32;
          umma_ss(x_tm, umma_desc_add(q_desc, off), umma_desc_add(kd, off), idesc_s, kk > 0);
        }
        umma_commit(&sm.r_s_full[r]);
      }
      __syncwarp();
    };

    if (ntiles > 0) issue_s(0);
    if (ntiles > 1) issue_s(1);
    for (uint32_t j = 0; j < ntiles; ++j) {
      const uint32_t g = tile_base + j;
      const uint32_t r = g % 3, ph = (g / 3) & 1, vs = g % 2, vph = (g / 2) & 1;
      mbar_wait(&sm.v_full[vs], vph, 640 + vs);
      mbar_wait(&sm.r_s_taken[r], ph, 650 + r);
      tc_fence_after();
      const uint32_t x_tm = tmem + dq_region_col(r);
      const uint64_t vd = v_kdesc0 + uint64_t(vs * SLOT16);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t off = (kk / 4) * SUB128 + (kk % 4) * 32;
          umma_ss(x_tm, umma_desc_add(do_desc, off), umma_desc_add(vd, off), idesc_s, kk > 0);
        }
        umma_commit(&sm.r_dp_full[r]);
        umma_commit(&sm.v_empty[vs]);
      }
      __syncwarp();
      if (j + 2 < ntiles) issue_s(j + 2);
    }
    umma_commit_w(&sm.qdo_empty);
    tile_base += ntiles;
  }
}

template <int D, bool BF16>
__device__ __forceinline__ void dq_issue_dq(DqSmem<D>& sm, const AttnBwdParams& p, uint32_t tmem_in) {
  constexpr uint32_t idesc_dq = umma_idesc_bf16(128, D, 0, 1, BF16 ? 1 : 0);
  constexpr uint64_t mnmaj = umma_smem_desc_hi_lo(SUB128, 1024, UMMA_LAYOUT_SW128);
  constexpr uint32_t SLOT16 = DqSmem<D>::TILE >> 4;
  const int lane = lane_id();
  const uint32_t tmem = warp_uniform(tmem_in);
  const uint32_t dq_tm = tmem + 256;
  uint32_t n_item = 0, tile_base = 0;
  const int total = dq_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DqItem it;
    dq_decode(p, idx, it);
    DqScan scan;
    dq_init_scan(scan, p, it);
    const uint32_t ntiles = scan.count(lane);
    const uint64_t k_mndesc0 = umma_desc(mnmaj, smem_u32(sm.k[0]));
    for (uint32_t j = 0; j < ntiles; ++j) {
      const uint32_t g = tile_base + j;
      const uint32_t r = g % 3, ph = (g / 3) & 1;
      mbar_wait(&sm.r_ds_ready[r], ph, 660 + r);
      if (j == 0) wait_acc_free(p, &sm.epi_done, &sm.carry_ready, n_item, 610);
      tc_fence_after();
      const uint32_t x_tm = tmem + dq_region_col(r);
      const uint64_t kmn = k_mndesc0 + uint64_t(r * SLOT16);
      const uint32_t acc0 = (j > 0 || p.carry_in) ? 1u : 0u;
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 128 / 16; ++kk) {
          umma_ts(dq_tm, x_tm + kk * 8, umma_desc_add(kmn, kk * 2048), idesc_dq, kk > 0 ? 1u : acc0);
        }
        umma_commit(&sm.k_empty[r]);
        umma_commit(&sm.r_free[r]);
      }
      __syncwarp();
    }
    if (ntiles == 0) wait_acc_free(p, &sm.epi_done, &sm.carry_ready, n_item, 612);
    umma_commit_w(&sm.dq_done);
    tile_base += ntiles;
  }
}

template <int D, bool BF16>
__device__ __forceinline__ void dq_softmax(DqSmem<D>& sm, const AttnBwdParams& p, const int W, uint32_t tmem) {
  const int wg_tid = threadIdx.x - 128 * W;
  const uint32_t lane_off = uint32_t((wg_tid / 32) * 32) << 16;
  const uint32_t dq_tm = tmem + 256 + lane_off;
  const int lane = lane_id();
  uint32_t n_item = 0, tile_base = 0;

  const bool clamp = p.softclamp > 0.f;
  const float mul = clamp ? 1.f : p.scale * kLog2e;
  const float pre = clamp ? p.scale / p.softclamp : 0.f;
  const float post = clamp ? p.softclamp * kLog2e : 0.f;

  const int total = dq_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DqItem it;
    dq_decode(p, idx, it);
    const int grow = it.row0 + wg_tid;
    const bool row_ok = grow < p.n_q;
    const int pos_q = pos_of(p.pos, p.rank, min(grow, p.n_q - 1)) + p.q_pos_offset;
    const size_t stat_row = ((size_t)(p.rank * 2) * p.batch * p.heads + (size_t)it.b * p.heads + it.h) * p.n_pad;
    float lse2 = INFINITY, delta = 0.f;
    if (row_ok) {
      lse2 = p.stat[stat_row + grow];
      delta = p.stat[stat_row + (size_t)p.batch * p.heads * p.n_pad + grow];
    }
    // hop mode: columns [W*D/2, (W+1)*D/2) of this row's dQ continue from the previous hop's launch (this thread
    // drained them in the previous item's epilogue)
    auto dq_row = [&]() { return (((size_t)it.b * p.n_q + (row_ok ? grow : 0)) * p.heads + it.h) * D + W * (D / 2); };
    if (p.carry_in) {
      carry_load<D / 2>(p.carry + dq_row(), row_ok, dq_tm + W * (D / 2));
      tc_fence_before();
      mbar_arrive(&sm.carry_ready);
    }

    DqScan scan;
    dq_init_scan(scan, p, it);
    ScanTile t;
    uint32_t jj = 0;
    while (scan.next(lane, t)) {
      const uint32_t jcur = jj++;
      if ((jcur & 1u) != (uint32_t)W) continue;
      // barriers of this tile are indexed by its TMEM region
      const uint32_t g = tile_base + jcur;
      const uint32_t r = g % 3;
      const uint32_t bpar = (g / 3) & 1;
      const uint32_t x_tm = tmem + dq_region_col(r) + lane_off;
      uint64_t* const b_s_full = &sm.r_s_full[r];
      uint64_t* const b_s_taken = &sm.r_s_taken[r];
      uint64_t* const b_dp_full = &sm.r_dp_full[r];
      uint64_t* const b_ds_ready = &sm.r_ds_ready[r];
      mbar_wait(b_s_full, bpar, 700 + W);
      tc_fence_after();
      uint32_t sr[128];
      tmem_ld32(x_tm + 0, sr + 0);
      tmem_ld32(x_tm + 32, sr + 32);
      tmem_ld32(x_tm + 64, sr + 64);
      tmem_ld32(x_tm + 96, sr + 96);
      tc_wait_ld();
      tc_fence_before();
      mbar_arrive(b_s_taken);

      if (t.part[0]) {
        const int c0 = t.idx * 128;
        const int split = p.pos.seg_len - c0;
        const int a0 = p.pos.base0[t.owner] + p.pos.stride * c0;
        const int a1 = p.pos.base1[t.owner] + p.pos.stride * (c0 - p.pos.seg_len);
        uint32_t mb[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        if (p.kmask_bits != nullptr) {
          const uint32_t* w = p.kmask_bits + ((size_t)t.owner * p.batch + it.b) * p.kmask_words + (size_t)t.idx * 4;
          mb[0] = w[0]; mb[1] = w[1]; mb[2] = w[2]; mb[3] = w[3];
        }
        const int ncols = p.n_k - c0;
#pragma unroll
        for (int j = 0; j < 128; ++j) {
          const int pk = (j < split ? a0 : a1) + p.pos.stride * j;
          bool keep = (j < ncols) && ((mb[j >> 5] >> (j & 31)) & 1u);
          if (p.causal) {
            keep = keep && (pk <= pos_q);
            if (p.window > 0) keep = keep && (pos_q - pk <= p.window);
          }
          if (!keep) sr[j] = 0xff800000u;
        }
      }

      // P = exp2(S*c - lse) while the tensor core is busy with dP = dO V^T of this tile (masked logits are
      // -inf and give exactly 0)
      if (!clamp) {
        const float2 mul2 = make_float2(mul, mul), nl2 = make_float2(-lse2, -lse2);
#pragma unroll
        for (int j = 0; j < 128; j += 2) {
          const float2 a = ffma2(make_float2(__uint_as_float(sr[j]), __uint_as_float(sr[j + 1])), mul2, nl2);
          const float2 e = make_float2(fast_exp2(a.x), fast_exp2(a.y));
          sr[j] = __float_as_uint(e.x);
          sr[j + 1] = __float_as_uint(e.y);
        }
      }
      mbar_wait(b_dp_full, bpar, 710 + W);
      tc_fence_after();
      // dS = P o (dP - delta) [* (1 - tanh^2) with softclamp]; the softmax scale is folded into the epilogue.
      if (!clamp) {
        uint32_t dpa[32], dpb[32];
        const float2 nd2 = make_float2(-delta, -delta);
        tmem_ld32(x_tm, dpa);
#pragma unroll
        for (int c = 0; c < 4; c += 2) {
          tc_wait_ld();
          tmem_ld32(x_tm + (c + 1) * 32, dpb);  // next chunk in flight during the math of this one
          {
            uint32_t w16[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 t = fadd2(make_float2(__uint_as_float(dpa[2 * i]), __uint_as_float(dpa[2 * i + 1])), nd2);
              const float2 dd = fmul2(make_float2(__uint_as_float(sr[c * 32 + 2 * i]), __uint_as_float(sr[c * 32 + 2 * i + 1])), t);
              w16[i] = BF16 ? pack_bf16x2(dd.x, dd.y) : pack_f16x2(dd.x, dd.y);
            }
            tc_wait_ld();  // chunk c+1 must have left TMEM before its columns are reused below
            if (c + 2 < 4) tmem_ld32(x_tm + (c + 2) * 32, dpa);
            tmem_st16(x_tm + c * 16, w16);
          }
          {
            uint32_t w16[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 t = fadd2(make_float2(__uint_as_float(dpb[2 * i]), __uint_as_float(dpb[2 * i + 1])), nd2);
              const float2 dd = fmul2(
                  make_float2(__uint_as_float(sr[(c + 1) * 32 + 2 * i]), __uint_as_float(sr[(c + 1) * 32 + 2 * i + 1])), t);
              w16[i] = BF16 ? pack_bf16x2(dd.x, dd.y) : pack_f16x2(dd.x, dd.y);
            }
            tmem_st16(x_tm + (c + 1) * 16, w16);
          }
        }
      } else {
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t dp[32];
          tmem_ld32(x_tm + c * 32, dp);
          tc_wait_ld();
          uint32_t w16[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float ds2[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              // dynamic chunk index: select the logit with a compile-time-indexed switch over the 4 chunks
              const int jj2 = 2 * i + e;
              float sv = __uint_as_float(sr[jj2]);
              if (c == 1) sv = __uint_as_float(sr[32 + jj2]);
              if (c == 2) sv = __uint_as_float(sr[64 + jj2]);
              if (c == 3) sv = __uint_as_float(sr[96 + jj2]);
              const float th = fast_tanh(sv * pre);
              float pj = fast_exp2(fmaf(th, post, -lse2));
              if (sv == -INFINITY) pj = 0.f;
              ds2[e] = pj * (__uint_as_float(dp[jj2]) - delta) * (1.f - th * th);
            }
            w16[i] = BF16 ? pack_bf16x2(ds2[0], ds2[1]) : pack_f16x2(ds2[0], ds2[1]);
          }
          tmem_st16(x_tm + c * 16, w16);
        }
      }
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(b_ds_ready);
    }
    tile_base += jj;

    // epilogue: warpgroup W converts columns [W*D/2, (W+1)*D/2) of dQ
    mbar_wait(&sm.dq_done, n_item & 1, 720 + W);
    tc_fence_after();
    if (p.carry_out) {
      // an item with no visible tile leaves a carried accumulator as it is
      if (jj > 0 || !p.carry_in) carry_store<D / 2>(p.carry + dq_row(), row_ok, jj > 0, dq_tm + W * (D / 2));
    } else {
      // the item may have had no visible tile at all: dQ is then zero (or the carry) and TMEM holds stale data
      const bool any = jj > 0 || p.carry_in;
      uint16_t* drow = reinterpret_cast<uint16_t*>(p.dq) + dq_row();
#pragma unroll
      for (int c = 0; c < D / 2; c += 32) {
        uint32_t acc[32];
        if (any) {
          tmem_ld32(dq_tm + W * (D / 2) + c, acc);
          tc_wait_ld();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = 0u;
        }
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a = __uint_as_float(acc[2 * i]) * p.scale, bq = __uint_as_float(acc[2 * i + 1]) * p.scale;
          w[i] = BF16 ? pack_bf16x2(a, bq) : pack_f16x2(a, bq);
        }
        if (row_ok) {
          uint4* dst = reinterpret_cast<uint4*>(drow + c);
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
        }
      }
    }
    tc_fence_before();
    mbar_arrive(&sm.epi_done);
  }
}

template <int D, bool BF16>
__global__ void __launch_bounds__(NTHREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_qd, const __grid_constant__ CUtensorMap map_kv,
                   const __grid_constant__ AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  DqSmem<D>& sm = *reinterpret_cast<DqSmem<D>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x / 32;
  if (threadIdx.x == 0) {
    mbar_init(&sm.qdo_full, 1);
    mbar_init(&sm.qdo_empty, 1);
    for (int i = 0; i < 3; ++i) {
      mbar_init(&sm.k_full[i], 1);
      mbar_init(&sm.k_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.v_full[i], 1);
      mbar_init(&sm.v_empty[i], 1);
    }
    for (int i = 0; i < 3; ++i) {
      mbar_init(&sm.r_s_full[i], 1);
      mbar_init(&sm.r_s_taken[i], 128);
      mbar_init(&sm.r_dp_full[i], 1);
      mbar_init(&sm.r_ds_ready[i], 128);
      mbar_init(&sm.r_free[i], 1);
    }
    mbar_init(&sm.dq_done, 1);
    mbar_init(&sm.epi_done, 256);
    mbar_init(&sm.carry_ready, 256);
    fence_mbar_init();
  }
  if (warp == 10) {
    tmem_alloc(&sm.tmem_base, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  if (warp >= 8) {  // control warps on the highest warp ids: the scheduler favours them
    setmaxnreg_dec<120>();
    if (warp == 8) dq_producer<D>(sm, p, &map_qd, &map_kv);
    if (warp == 9) dq_issue_sdp<D, BF16>(sm, p, tmem);
    if (warp == 10) dq_issue_dq<D, BF16>(sm, p, tmem);
  } else {
    setmaxnreg_inc<192>();
    dq_softmax<D, BF16>(sm, p, warp < 4 ? 0 : 1, tmem);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) tmem_dealloc(tmem, 512);
}

// =================================================================================================
// dK/dV kernel
// =================================================================================================
constexpr int QSTAGES = 4;

template <int D>
struct DkvSmem {
  static constexpr int NSUB = D / 64;
  static constexpr int KV_TILE = NSUB * SUB128;  // 128 keys
  static constexpr int Q_TILE = NSUB * SUB64;    // 64 queries
  alignas(1024) uint8_t k[KV_TILE];
  alignas(1024) uint8_t v[KV_TILE];
  alignas(1024) uint8_t q[QSTAGES][Q_TILE];
  alignas(1024) uint8_t dout[QSTAGES][Q_TILE];
  alignas(16) float lse2[QSTAGES][64];
  alignas(16) float delta[QSTAGES][64];
  uint64_t kv_full, kv_empty;
  uint64_t qd_full[QSTAGES], qd_empty[QSTAGES];
  uint64_t s_full[2], s_free[2], dp_full[2], pds_ready[2];
  uint64_t acc_done, epi_done;
  uint64_t carry_ready;  // hop mode: both warpgroups have loaded the item's carried dK / dV into TMEM
  uint32_t tmem_base;
};

struct DkvItem {
  int b, kvh, kt, key0;
  int klo, khi;
  bool k_tail;
};

__device__ __forceinline__ int dkv_num_items(const AttnBwdParams& p) {
  return p.batch * p.kv_heads * ((p.n_k + 127) / 128);
}

__device__ __forceinline__ void dkv_decode(const AttnBwdParams& p, int idx, DkvItem& it) {
  const int bh = p.batch * p.kv_heads;
  it.kt = idx / bh;  // early key tiles are visible to the most queries under causal masking: heaviest first
  const int r = idx % bh;
  it.b = r / p.kv_heads;
  it.kvh = r % p.kv_heads;
  it.key0 = it.kt * 128;
  pos_range(p.pos, p.rank, it.key0, min(it.key0 + 128, p.n_k) - 1, it.klo, it.khi);
  it.k_tail = (it.key0 + 128) > p.n_k;
}

using DkvScan = WarpTileScan<1, true>;

// streamed side = query tiles of 64 rows; rep = index of the query head inside the GQA group
__device__ __forceinline__ void dkv_init_scan(DkvScan& sc, const AttnBwdParams& p, const DkvItem& it) {
  sc.pm = &p.pos;
  sc.hop_owner = p.hop_owner;
  sc.hop_count = p.hop_count;
  sc.groups = p.heads / p.kv_heads;
  sc.n_stream = p.n_q;
  sc.tile = 64;
  sc.stream_off = p.q_pos_offset;
  sc.stat_off = 0;
  sc.mc = MaskCfg{p.causal, p.window, p.kmask_bits != nullptr};
  sc.st[0] = StatRange{it.klo, it.khi, true, it.k_tail};
}

template <int D>
__device__ __forceinline__ void dkv_producer(DkvSmem<D>& sm, const AttnBwdParams& p, const CUtensorMap* map_qd64,
                                             const CUtensorMap* map_kv) {
  constexpr int NSUB = DkvSmem<D>::NSUB;
  constexpr uint32_t KV_TILE = DkvSmem<D>::KV_TILE, Q_TILE = DkvSmem<D>::Q_TILE;
  const int lane = lane_id();
  uint32_t n_item = 0, n_tile = 0;
  uint32_t ready_mask = 1u << p.rank;
  const int total = dkv_num_items(p);
  const size_t stat_half = (size_t)p.batch * p.heads * p.n_pad;
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DkvItem it;
    dkv_decode(p, idx, it);
    if (lane == 0) {
      mbar_wait(&sm.kv_empty, (n_item & 1) ^ 1, 800);
      mbar_expect_tx(&sm.kv_full, 2 * KV_TILE);
#pragma unroll
      for (int s = 0; s < NSUB; ++s) {
        tma_load_4d(sm.k + s * SUB128, map_kv, &sm.kv_full, s * 64, it.key0, it.b * p.kv_heads + it.kvh,
                    p.rank * 2);
        tma_load_4d(sm.v + s * SUB128, map_kv, &sm.kv_full, s * 64, it.key0, it.b * p.kv_heads + it.kvh,
                    p.rank * 2 + 1);
      }
    }
    DkvScan scan;
    dkv_init_scan(scan, p, it);
    ScanTile t;
    while (scan.next(lane, t)) {
      if (lane == 0) {
        wait_owner_ready(p, t.owner, ready_mask, 801);
        const uint32_t st = n_tile % QSTAGES, ph = (n_tile / QSTAGES) & 1;
        const int h = t.rep * p.kv_heads + it.kvh;
        const int bh = it.b * p.heads + h;
        mbar_wait(&sm.qd_empty[st], ph ^ 1, 810 + st);
        mbar_expect_tx(&sm.qd_full[st], 2 * Q_TILE + 2 * 64 * 4);
#pragma unroll
        for (int s = 0; s < NSUB; ++s) {
          tma_load_4d(sm.q[st] + s * SUB64, map_qd64, &sm.qd_full[st], s * 64, t.idx * 64, bh, t.owner * 2);
          tma_load_4d(sm.dout[st] + s * SUB64, map_qd64, &sm.qd_full[st], s * 64, t.idx * 64, bh, t.owner * 2 + 1);
        }
        const float* srow = p.stat + ((size_t)(t.owner * 2) * p.batch * p.heads + bh) * p.n_pad + (size_t)t.idx * 64;
        bulk_load_1d(sm.lse2[st], srow, 64 * 4, &sm.qd_full[st]);
        bulk_load_1d(sm.delta[st], srow + stat_half, 64 * 4, &sm.qd_full[st]);
      }
      n_tile++;
      __syncwarp();
    }
  }
}

// Two issuing warps.  Profiling the first, single-issuer version of this kernel showed the MMA-issuing warp executing ~380
// instructions of polling / bookkeeping per 128 x 64 step while the tensor pipe back-pressured it only 10 % of the time:
// the issuer's own control flow, not the tensor core, paced the kernel.  Here the work is split by TMEM block instead of
// by stream, which makes every wait a plain blocking mbarrier wait in program order (no state machine, no scanner in
// the issuers, just the tile count of the item):
//   warp 9  "S issuer"   : S^T(j) into X_w                       gated by qd_full(stage j), s_free[w]
//   warp 10 "acc issuer" : dP^T(j) into Y_w, dV/dK(j) from Y_w   gated by qd_full(stage j), pds_ready[w]
// The two warps never touch the same TMEM block, and only warp 10 accumulates into dK/dV, so no cross-warp ordering of
// tcgen05.mma is relied upon.
template <int D, bool BF16>
__device__ __forceinline__ void dkv_issue_s(DkvSmem<D>& sm, const AttnBwdParams& p, uint32_t tmem_in) {
  constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64, 0, 0, BF16 ? 1 : 0);
  constexpr uint64_t kmaj = umma_smem_desc_hi_lo(16, 1024, UMMA_LAYOUT_SW128);
  constexpr uint32_t STAGE16 = DkvSmem<D>::Q_TILE >> 4;
  const int lane = lane_id();
  const uint32_t tmem = warp_uniform(tmem_in);
  uint32_t n_item = 0, tile_base = 0;
  uint32_t c_s[2] = {0, 0};  // S^T issued per stream (cumulative): s_free parity
  const int total = dkv_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DkvItem it;
    dkv_decode(p, idx, it);
    DkvScan scan;
    dkv_init_scan(scan, p, it);
    const uint32_t ntiles = scan.count(lane);
    mbar_wait(&sm.kv_full, n_item & 1, 900);
    tc_fence_after();
    const uint64_t k_desc = umma_desc(kmaj, smem_u32(sm.k));
    const uint64_t q_kdesc0 = umma_desc(kmaj, smem_u32(sm.q[0]));
    for (uint32_t j = 0; j < ntiles; ++j) {
      const uint32_t w = j & 1u;
      const uint32_t g = tile_base + j;
      const uint32_t st = g % QSTAGES, ph = (g / QSTAGES) & 1;
      mbar_wait(&sm.qd_full[st], ph, 920 + st);
      // X_w is free once S^T has been pulled into registers
      if (c_s[w] > 0) mbar_wait(&sm.s_free[w], (c_s[w] - 1u) & 1, 930 + w);
      tc_fence_after();
      const uint32_t x_tm = tmem + w * 128u;
      const uint64_t qk = q_kdesc0 + uint64_t(st * STAGE16);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t offk = (kk / 4) * SUB128 + (kk % 4) * 32;
          const uint32_t offq = (kk / 4) * SUB64 + (kk % 4) * 32;
          umma_ss(x_tm, umma_desc_add(k_desc, offk), umma_desc_add(qk, offq), idesc_s, kk > 0);
        }
        umma_commit(&sm.s_full[w]);
      }
      __syncwarp();
      c_s[w]++;
    }
    umma_commit_w(&sm.kv_empty);  // second arrival comes from the acc issuer
    tile_base += ntiles;
  }
}

template <int D, bool BF16>
__device__ __forceinline__ void dkv_issue_acc(DkvSmem<D>& sm, const AttnBwdParams& p, uint32_t tmem_in) {
  constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64, 0, 0, BF16 ? 1 : 0);
  constexpr uint32_t idesc_acc = umma_idesc_bf16(128, D, 0, 1, BF16 ? 1 : 0);
  constexpr uint64_t kmaj = umma_smem_desc_hi_lo(16, 1024, UMMA_LAYOUT_SW128);
  constexpr uint64_t mnmaj64 = umma_smem_desc_hi_lo(SUB64, 1024, UMMA_LAYOUT_SW128);
  constexpr uint32_t STAGE16 = DkvSmem<D>::Q_TILE >> 4;
  const int lane = lane_id();
  const uint32_t tmem = warp_uniform(tmem_in);
  const uint32_t dk_tm = tmem + 256, dv_tm = tmem + 256 + D;
  uint32_t n_item = 0, tile_base = 0;
  uint32_t c_b[2] = {0, 0};  // dV/dK issued per stream (cumulative): pds_ready parity
  const int total = dkv_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DkvItem it;
    dkv_decode(p, idx, it);
    DkvScan scan;
    dkv_init_scan(scan, p, it);
    const uint32_t ntiles = scan.count(lane);
    mbar_wait(&sm.kv_full, n_item & 1, 901);
    tc_fence_after();
    const uint64_t v_desc = umma_desc(kmaj, smem_u32(sm.v));
    const uint64_t do_kdesc0 = umma_desc(kmaj, smem_u32(sm.dout[0]));
    const uint64_t q_mndesc0 = umma_desc(mnmaj64, smem_u32(sm.q[0]));
    const uint64_t do_mndesc0 = umma_desc(mnmaj64, smem_u32(sm.dout[0]));

    auto issue_dp = [&](uint32_t j) {  // dP^T(j) = V dO^T into Y_w (free: dV/dK(j-2) precede it in this warp's FIFO)
      const uint32_t w = j & 1u;
      const uint32_t g = tile_base + j;
      const uint32_t st = g % QSTAGES, ph = (g / QSTAGES) & 1;
      mbar_wait(&sm.qd_full[st], ph, 924 + st);
      tc_fence_after();
      const uint32_t y_tm = tmem + w * 128u + 64u;
      const uint64_t dok = do_kdesc0 + uint64_t(st * STAGE16);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t offk = (kk / 4) * SUB128 + (kk % 4) * 32;
          const uint32_t offq = (kk / 4) * SUB64 + (kk % 4) * 32;
          umma_ss(y_tm, umma_desc_add(v_desc, offk), umma_desc_add(dok, offq), idesc_s, kk > 0);
        }
        umma_commit(&sm.dp_full[w]);
      }
      __syncwarp();
    };

    if (ntiles > 0) issue_dp(0);
    if (ntiles > 1) issue_dp(1);
    for (uint32_t j = 0; j < ntiles; ++j) {
      const uint32_t w = j & 1u;
      const uint32_t st = (tile_base + j) % QSTAGES;
      mbar_wait(&sm.pds_ready[w], c_b[w] & 1, 940 + w);
      if (j == 0) wait_acc_free(p, &sm.epi_done, &sm.carry_ready, n_item, 910);
      tc_fence_after();
      const uint32_t y_tm = tmem + w * 128u + 64u;
      const uint64_t qmn = q_mndesc0 + uint64_t(st * STAGE16), domn = do_mndesc0 + uint64_t(st * STAGE16);
      const uint32_t acc0 = (j > 0 || p.carry_in) ? 1u : 0u;
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 64 / 16; ++kk) {
          umma_ts(dv_tm, y_tm + kk * 8, umma_desc_add(domn, kk * 2048), idesc_acc, kk > 0 ? 1u : acc0);
        }
#pragma unroll
        for (int kk = 0; kk < 64 / 16; ++kk) {
          umma_ts(dk_tm, y_tm + 32 + kk * 8, umma_desc_add(qmn, kk * 2048), idesc_acc, kk > 0 ? 1u : acc0);
        }
        umma_commit(&sm.qd_empty[st]);
      }
      __syncwarp();
      c_b[w]++;
      if (j + 2 < ntiles) issue_dp(j + 2);
    }
    if (ntiles == 0) wait_acc_free(p, &sm.epi_done, &sm.carry_ready, n_item, 912);
    umma_commit_w(&sm.acc_done);
    umma_commit_w(&sm.kv_empty);
    tile_base += ntiles;
  }
}

template <int D, bool BF16>
__device__ __forceinline__ void dkv_softmax(DkvSmem<D>& sm, const AttnBwdParams& p, const int W, uint32_t tmem) {
  const int wg_tid = threadIdx.x - 128 * W;
  const uint32_t lane_off = uint32_t((wg_tid / 32) * 32) << 16;
  const uint32_t st_tm = tmem + W * 128 + lane_off;
  const uint32_t dpt_tm = tmem + W * 128 + 64 + lane_off;
  const int lane = lane_id();
  uint32_t cnt = 0, n_item = 0, tile_base = 0;

  const bool clamp = p.softclamp > 0.f;
  const float mul = clamp ? 1.f : p.scale * kLog2e;
  const float pre = clamp ? p.scale / p.softclamp : 0.f;
  const float post = clamp ? p.softclamp * kLog2e : 0.f;

  const int total = dkv_num_items(p);
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x, ++n_item) {
    DkvItem it;
    dkv_decode(p, idx, it);
    const int key = it.key0 + wg_tid;
    bool key_ok = key < p.n_k;
    const int pos_k = pos_of(p.pos, p.rank, min(key, p.n_k - 1));
    if (key_ok && p.kmask_bits != nullptr) {
      const uint32_t wbits = p.kmask_bits[((size_t)p.rank * p.batch + it.b) * p.kmask_words + (key >> 5)];
      key_ok = (wbits >> (key & 31)) & 1u;
    }
    // warpgroup 0 owns dK, warpgroup 1 dV: in hop mode this key's row continues from the previous hop's launch (this
    // thread drained it in the previous item's epilogue)
    auto carry_row = [&]() {
      return p.carry + (size_t)W * p.batch * p.n_k * p.kv_heads * D +
             (((size_t)it.b * p.n_k + (key < p.n_k ? key : 0)) * p.kv_heads + it.kvh) * D;
    };
    if (p.carry_in) {
      carry_load<D>(carry_row(), key < p.n_k, tmem + 256 + (W == 0 ? 0 : D) + lane_off);
      tc_fence_before();
      mbar_arrive(&sm.carry_ready);
    }

    DkvScan scan;
    dkv_init_scan(scan, p, it);
    ScanTile t;
    uint32_t jn = 0;
    while (scan.next(lane, t)) {
      const uint32_t jj = jn++;
      if ((jj & 1u) != (uint32_t)W) continue;
      const uint32_t stg = (tile_base + jj) % QSTAGES;
      uint32_t sr[64], dp[64];
      mbar_wait((&sm.s_full[0] + W), cnt & 1, 1000 + W);
      tc_fence_after();
      tmem_ld32(st_tm + 0, sr + 0);
      tmem_ld32(st_tm + 32, sr + 32);
      tc_wait_ld();
      tc_fence_before();
      mbar_arrive((&sm.s_free[0] + W));  // X_w may take S^T of this stream's next tile now

      const int c0 = t.idx * 64;
      const float4* l4 = reinterpret_cast<const float4*>(sm.lse2[stg]);
      const float4* d4 = reinterpret_cast<const float4*>(sm.delta[stg]);
      uint32_t pw[32], dw[32];
      // P^T = exp2(S^T * c - lse[col]); dS^T = P^T o (dP^T - delta[col]).  The softmax scale is folded into the dK
      // epilogue.  The fast path has no per-element predicate at all; ragged / diagonal / padded tiles and the
      // softclamp variant take the general path.
      if (!t.part[0] && !clamp) {
#pragma unroll
        for (int q4 = 0; q4 < 16; ++q4) {
          const float4 lv = l4[q4];
          const float2 mul2 = make_float2(mul, mul);
          const float2 a01 = ffma2(make_float2(__uint_as_float(sr[q4 * 4 + 0]), __uint_as_float(sr[q4 * 4 + 1])), mul2,
                                   make_float2(-lv.x, -lv.y));
          const float2 a23 = ffma2(make_float2(__uint_as_float(sr[q4 * 4 + 2]), __uint_as_float(sr[q4 * 4 + 3])), mul2,
                                   make_float2(-lv.z, -lv.w));
          const float p0 = fast_exp2(a01.x), p1 = fast_exp2(a01.y), p2 = fast_exp2(a23.x), p3 = fast_exp2(a23.y);
          sr[q4 * 4 + 0] = __float_as_uint(p0);
          sr[q4 * 4 + 1] = __float_as_uint(p1);
          sr[q4 * 4 + 2] = __float_as_uint(p2);
          sr[q4 * 4 + 3] = __float_as_uint(p3);
          pw[q4 * 2] = BF16 ? pack_bf16x2(p0, p1) : pack_f16x2(p0, p1);
          pw[q4 * 2 + 1] = BF16 ? pack_bf16x2(p2, p3) : pack_f16x2(p2, p3);
        }
        mbar_wait((&sm.dp_full[0] + W), cnt & 1, 1004 + W);
        tc_fence_after();
        tmem_ld32(dpt_tm + 0, dp + 0);
        tmem_ld32(dpt_tm + 32, dp + 32);
        tc_wait_ld();  // dP^T has landed
#pragma unroll
        for (int q4 = 0; q4 < 16; ++q4) {
          const float4 dv = d4[q4];
          const float2 t01 = fadd2(make_float2(__uint_as_float(dp[q4 * 4 + 0]), __uint_as_float(dp[q4 * 4 + 1])),
                                   make_float2(-dv.x, -dv.y));
          const float2 t23 = fadd2(make_float2(__uint_as_float(dp[q4 * 4 + 2]), __uint_as_float(dp[q4 * 4 + 3])),
                                   make_float2(-dv.z, -dv.w));
          const float2 e01 = fmul2(make_float2(__uint_as_float(sr[q4 * 4 + 0]), __uint_as_float(sr[q4 * 4 + 1])), t01);
          const float2 e23 = fmul2(make_float2(__uint_as_float(sr[q4 * 4 + 2]), __uint_as_float(sr[q4 * 4 + 3])), t23);
          dw[q4 * 2] = BF16 ? pack_bf16x2(e01.x, e01.y) : pack_f16x2(e01.x, e01.y);
          dw[q4 * 2 + 1] = BF16 ? pack_bf16x2(e23.x, e23.y) : pack_f16x2(e23.x, e23.y);
        }
      } else {
        mbar_wait((&sm.dp_full[0] + W), cnt & 1, 1004 + W);
        tc_fence_after();
        tmem_ld32(dpt_tm + 0, dp + 0);
        tmem_ld32(dpt_tm + 32, dp + 32);
        tc_wait_ld();  // dP^T has landed
        const int split = p.pos.seg_len - c0;
        const int a0 = p.pos.base0[t.owner] + p.pos.stride * c0 + p.q_pos_offset;
        const int a1 = p.pos.base1[t.owner] + p.pos.stride * (c0 - p.pos.seg_len) + p.q_pos_offset;
        const int ncols = p.n_q - c0;
        const bool part = t.part[0];
#pragma unroll
        for (int q4 = 0; q4 < 16; ++q4) {
          const float4 lv = l4[q4];
          const float4 dv = d4[q4];
          const float ls[4] = {lv.x, lv.y, lv.z, lv.w};
          const float dl[4] = {dv.x, dv.y, dv.z, dv.w};
          float pp[4], dd[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = q4 * 4 + e;
            const float sv = __uint_as_float(sr[j]);
            float pj, chain = 1.f;
            if (clamp) {
              const float th = fast_tanh(sv * pre);
              pj = fast_exp2(fmaf(th, post, -ls[e]));
              chain = 1.f - th * th;
            } else {
              pj = fast_exp2(fmaf(sv, mul, -ls[e]));
            }
            bool keep = true;
            if (part) {
              const int pq = (j < split ? a0 : a1) + p.pos.stride * j;
              keep = key_ok && (j < ncols);
              if (p.causal) {
                keep = keep && (pos_k <= pq);
                if (p.window > 0) keep = keep && (pq - pos_k <= p.window);
              }
            }
            if (!keep) pj = 0.f;
            pp[e] = pj;
            dd[e] = pj * (__uint_as_float(dp[j]) - dl[e]) * chain;
          }
          pw[q4 * 2] = BF16 ? pack_bf16x2(pp[0], pp[1]) : pack_f16x2(pp[0], pp[1]);
          pw[q4 * 2 + 1] = BF16 ? pack_bf16x2(pp[2], pp[3]) : pack_f16x2(pp[2], pp[3]);
          dw[q4 * 2] = BF16 ? pack_bf16x2(dd[0], dd[1]) : pack_f16x2(dd[0], dd[1]);
          dw[q4 * 2 + 1] = BF16 ? pack_bf16x2(dd[2], dd[3]) : pack_f16x2(dd[2], dd[3]);
        }
      }
      // P^T | dS^T share the dP^T block; the S^T block already belongs to the next tile
      tmem_st32(dpt_tm, pw);
      tmem_st32(dpt_tm + 32, dw);
      tc_wait_st();
      tc_fence_before();
      mbar_arrive((&sm.pds_ready[0] + W));
      cnt++;
    }
    tile_base += jn;  // both warpgroups walk the whole sequence, so the stage ring stays in step

    // epilogue: warpgroup 0 writes dK, warpgroup 1 writes dV
    mbar_wait(&sm.acc_done, n_item & 1, 1010 + W);
    tc_fence_after();
    const bool row_ok = key < p.n_k;
    const uint32_t acc_tm = tmem + 256 + (W == 0 ? 0 : D) + lane_off;
    if (p.carry_out) {
      // an item with no visible tile leaves a carried accumulator as it is
      if (jn > 0 || !p.carry_in) carry_store<D>(carry_row(), row_ok, jn > 0, acc_tm);
    } else {
      const bool any = jn > 0 || p.carry_in;
      uint16_t* out = reinterpret_cast<uint16_t*>(W == 0 ? p.dk : p.dv) +
                      (((size_t)it.b * p.n_k + (row_ok ? key : 0)) * p.kv_heads + it.kvh) * D;
#pragma unroll
      for (int c = 0; c < D; c += 32) {
        uint32_t acc[32];
        if (any) {
          tmem_ld32(acc_tm + c, acc);
          tc_wait_ld();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = 0u;
        }
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float osc = W == 0 ? p.scale : 1.f;  // dK carries the folded softmax scale
          const float a = __uint_as_float(acc[2 * i]) * osc, bq = __uint_as_float(acc[2 * i + 1]) * osc;
          w[i] = BF16 ? pack_bf16x2(a, bq) : pack_f16x2(a, bq);
        }
        if (row_ok) {
          uint4* dst = reinterpret_cast<uint4*>(out + c);
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
        }
      }
    }
    tc_fence_before();
    mbar_arrive(&sm.epi_done);
  }
}

template <int D, bool BF16>
__global__ void __launch_bounds__(NTHREADS, 1)
attn_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap map_qd64, const __grid_constant__ CUtensorMap map_kv,
                     const __grid_constant__ AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  DkvSmem<D>& sm = *reinterpret_cast<DkvSmem<D>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x / 32;
  if (threadIdx.x == 0) {
    mbar_init(&sm.kv_full, 1);
    mbar_init(&sm.kv_empty, 2);
    for (int i = 0; i < QSTAGES; ++i) {
      mbar_init(&sm.qd_full[i], 1);
      mbar_init(&sm.qd_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.pds_ready[i], 128);
      mbar_init(&sm.s_full[i], 1);
      mbar_init(&sm.s_free[i], 128);
      mbar_init(&sm.dp_full[i], 1);
    }
    mbar_init(&sm.acc_done, 1);
    mbar_init(&sm.epi_done, 256);
    mbar_init(&sm.carry_ready, 256);
    fence_mbar_init();
  }
  if (warp == 10) {
    tmem_alloc(&sm.tmem_base, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  if (warp >= 8) {  // control warps on the highest warp ids: the scheduler favours them
    setmaxnreg_dec<120>();
    if (warp == 8) dkv_producer<D>(sm, p, &map_qd64, &map_kv);
    if (warp == 9) dkv_issue_s<D, BF16>(sm, p, tmem);
    if (warp == 10) dkv_issue_acc<D, BF16>(sm, p, tmem);
  } else {
    setmaxnreg_inc<192>();
    dkv_softmax<D, BF16>(sm, p, warp < 4 ? 0 : 1, tmem);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) tmem_dealloc(tmem, 512);
}

// =================================================================================================
// prep: delta = rowsum(o * do), lse -> log2 domain, q / do -> head-major slot
// =================================================================================================
template <bool BF16>
__global__ void bwd_prep_kernel(const uint16_t* __restrict__ q, const uint16_t* __restrict__ o,
                                const uint16_t* __restrict__ dout, const float* __restrict__ lse,
                                uint16_t* __restrict__ qdo_slot, float* __restrict__ stat_slot, int batch, int n,
                                int heads, int d, int n_pad) {
  const int vec_per_row = d / 8;  // 8 or 16 lanes per row
  const long long rows = (long long)batch * n * heads;
  const long long gid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long row = gid / vec_per_row;
  const int c = gid % vec_per_row;
  float part = 0.f;
  long long out_row = 0;
  int hh = 0, i = 0, b = 0;
  const bool active = row < rows;
  if (active) {
    hh = row % heads;
    i = (row / heads) % n;
    b = row / ((long long)heads * n);
    out_row = ((long long)b * heads + hh) * n + i;
    const uint4 qv = reinterpret_cast<const uint4*>(q + row * d)[c];
    const uint4 ov = reinterpret_cast<const uint4*>(o + row * d)[c];
    const uint4 dv = reinterpret_cast<const uint4*>(dout + row * d)[c];
    reinterpret_cast<uint4*>(qdo_slot + out_row * d)[c] = qv;
    reinterpret_cast<uint4*>(qdo_slot + (rows + out_row) * d)[c] = dv;
    const uint32_t ow[4] = {ov.x, ov.y, ov.z, ov.w}, dw[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float o0, o1, d0, d1;
      if (BF16) {
        o0 = __uint_as_float(ow[e] << 16); o1 = __uint_as_float(ow[e] & 0xffff0000u);
        d0 = __uint_as_float(dw[e] << 16); d1 = __uint_as_float(dw[e] & 0xffff0000u);
      } else {
        const __half2 oh = *reinterpret_cast<const __half2*>(&ow[e]);
        const __half2 dh = *reinterpret_cast<const __half2*>(&dw[e]);
        o0 = __low2float(oh); o1 = __high2float(oh);
        d0 = __low2float(dh); d1 = __high2float(dh);
      }
      part += o0 * d0 + o1 * d1;
    }
  }
  for (int off = vec_per_row / 2; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
  if (active && c == 0) {
    const long long srow = ((long long)b * heads + hh) * n_pad + i;
    const float l = lse[((long long)b * heads + hh) * n + i];
    stat_slot[srow] = l * kLog2e;  // +inf stays +inf
    stat_slot[(long long)batch * heads * n_pad + srow] = part;
  }
}

}  // namespace

template <int D>
void launch_attn_bwd_dq(const CUtensorMap& map_qd, const CUtensorMap& map_kv, const AttnBwdParams& p, int num_sms,
                        cudaStream_t stream) {
  using Kern = void (*)(const CUtensorMap, const CUtensorMap, const AttnBwdParams);
  Kern kern = p.is_bf16 ? attn_bwd_dq_kernel<D, true> : attn_bwd_dq_kernel<D, false>;
  const size_t smem = sizeof(DqSmem<D>) + 1024;
  cuda_check(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "bwd_dq smem attr");
  const int items = p.batch * p.heads * ((p.n_q + 127) / 128);
  const int grid = items < num_sms ? items : num_sms;
  void* args[] = {(void*)&map_qd, (void*)&map_kv, (void*)&p};
  cuda_check(cudaLaunchKernel((void*)kern, dim3(grid), dim3(NTHREADS), args, smem, stream), "bwd_dq launch");
}

template <int D>
void launch_attn_bwd_dkdv(const CUtensorMap& map_qd64, const CUtensorMap& map_kv, const AttnBwdParams& p,
                          int num_sms, cudaStream_t stream) {
  using Kern = void (*)(const CUtensorMap, const CUtensorMap, const AttnBwdParams);
  Kern kern = p.is_bf16 ? attn_bwd_dkdv_kernel<D, true> : attn_bwd_dkdv_kernel<D, false>;
  const size_t smem = sizeof(DkvSmem<D>) + 1024;
  cuda_check(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
             "bwd_dkdv smem attr");
  const int items = p.batch * p.kv_heads * ((p.n_k + 127) / 128);
  const int grid = items < num_sms ? items : num_sms;
  void* args[] = {(void*)&map_qd64, (void*)&map_kv, (void*)&p};
  cuda_check(cudaLaunchKernel((void*)kern, dim3(grid), dim3(NTHREADS), args, smem, stream), "bwd_dkdv launch");
}

void launch_bwd_prep(const void* q, const void* o, const void* dout, const float* lse, void* qdo_slot,
                     float* stat_slot, int batch, int n, int heads, int d, int n_pad, int is_bf16,
                     cudaStream_t stream) {
  const long long threads_total = (long long)batch * n * heads * (d / 8);
  if (threads_total == 0) return;
  const int threads = 256;
  const long long blocks = (threads_total + threads - 1) / threads;
  auto kern = is_bf16 ? bwd_prep_kernel<true> : bwd_prep_kernel<false>;
  kern<<<(unsigned)blocks, threads, 0, stream>>>(
      reinterpret_cast<const uint16_t*>(q), reinterpret_cast<const uint16_t*>(o),
      reinterpret_cast<const uint16_t*>(dout), lse, reinterpret_cast<uint16_t*>(qdo_slot), stat_slot, batch, n, heads,
      d, n_pad);
  cuda_check(cudaGetLastError(), "bwd_prep launch");
}

template void launch_attn_bwd_dq<64>(const CUtensorMap&, const CUtensorMap&, const AttnBwdParams&, int, cudaStream_t);
template void launch_attn_bwd_dq<128>(const CUtensorMap&, const CUtensorMap&, const AttnBwdParams&, int, cudaStream_t);
template void launch_attn_bwd_dkdv<64>(const CUtensorMap&, const CUtensorMap&, const AttnBwdParams&, int, cudaStream_t);
template void launch_attn_bwd_dkdv<128>(const CUtensorMap&, const CUtensorMap&, const AttnBwdParams&, int, cudaStream_t);

}  // namespace rab
