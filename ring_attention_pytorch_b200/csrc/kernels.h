// Plain C++/CUDA launch API shared between the .cu kernels and the torch bindings.
// Nothing in here depends on torch headers, so kernels rebuild in seconds.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tmap.h"

namespace rab {

constexpr int kMaxWorld = 16;

// ------------------------------------------------------------------------------------------------
// descriptor probe (tests)
// ------------------------------------------------------------------------------------------------
struct ProbeParams {
  int mode;  // 0: SS K-major x K-major, 1: SS with MN-major B, 2: TS (A in TMEM) with MN-major B
  int n;     // MMA N
  int k;     // reduction length (multiple of 16, <= 128)
  uint32_t idesc;
  uint32_t a_lbo, a_sbo;
  uint32_t b_lbo, b_sbo;
  uint32_t b_kstep_bytes;  // start-address advance per K=16 step for an MN-major B operand
};
void launch_umma_probe(const CUtensorMap& map_a, const CUtensorMap& map_b, const ProbeParams& p,
                       const void* a_raw, float* out, cudaStream_t stream);
void launch_umma_rate(int mode, int n, int reps, int alt, int ctas, long long* out, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// position maps: how local index i on ring rank r maps to a global token position.
//   i <  seg_len : base0[r] + stride * i
//   i >= seg_len : base1[r] + stride * (i - seg_len)
// plain ring   : seg_len = n, base0 = r*n,  stride = 1
// striped ring : seg_len = n, base0 = r,    stride = W
// zig-zag      : seg_len = n/2, base0 = r*c, base1 = (2W-1-r)*c, stride = 1
// ------------------------------------------------------------------------------------------------
struct PosMap {
  int stride;
  int seg_len;
  int base0[kMaxWorld];
  int base1[kMaxWorld];
};

// ------------------------------------------------------------------------------------------------
// the attention problem the forward and both backwards share (one ring rank's view of it)
// ------------------------------------------------------------------------------------------------
struct AttnProblem {
  int batch, heads, kv_heads;
  int n_q;      // local query rows
  int n_k;      // keys per owner slot
  int world;    // number of KV owner slots (ring size)
  int rank;     // ring-local rank of this device
  int causal;
  int window;   // max (pos_q - pos_k), <= 0 disables
  int is_bf16;
  float scale;        // softmax scale
  float softclamp;    // 0 disables, else tanh clamp value applied to scaled logits
  PosMap pos;
  int q_pos_offset;   // added to query positions (cross-attention causal alignment)
  int hop_count;
  int hop_owner[kMaxWorld];  // owners visited; hop 0 is this rank unless the launch covers one hop only
  // key-padding bits: [world][batch][kmask_words] uint32 (bit set = keep), may be null
  const uint32_t* kmask_bits;
  int kmask_words;
};

// ------------------------------------------------------------------------------------------------
// fused ring flash-attention forward
// ------------------------------------------------------------------------------------------------
struct AttnFwdParams : AttnProblem {
  // outputs
  void* o;       // [b, n_q, h, d] 16-bit
  float* lse;    // [b, h, n_q] natural-log lse (+inf for rows with no visible key)
  // in-kernel K/V gather over NVLink
  uint8_t* kv_local;                  // this rank's [world][2][b*hk][n_k][d] buffer
  const uint8_t* kv_peer[kMaxWorld];  // kv_peer[o]: owner o's own [2][b*hk][n_k][d] slot (peer-mapped)
  unsigned long long slot_bytes;      // bytes of one owner slot (K and V)
  uint32_t* ready;                    // [world] arrival counters, zero before launch
  unsigned long long* fetch_times;    // optional [gridDim][2] globaltimer ns: first / last activity of each CTA's fetcher
  // hop-at-a-time mode (memory = "ring"): one launch per ring hop, the online-softmax state travels between launches
  float* carry_o;    // fp32 [b, n_q, h, d] un-normalised O (in / out), null = single-launch mode
  float* carry_ml;   // fp32 [2][b*h][n_q]: running maximum (scaled log2 domain) and running sum
  int carry_in;      // 1: initialise O / m / l of every item from the carry buffers
  int carry_out;     // 1: store the un-normalised state instead of the final O / lse
  int all_ready;     // 1: every slot this launch reads is already complete (no in-kernel fetch, no ready flags)
};

template <int D>
void launch_attn_fwd(const CUtensorMap& map_q, const CUtensorMap& map_kv, const AttnFwdParams& p, int num_sms,
                     cudaStream_t stream);
size_t attn_fwd_smem_bytes(int head_dim);

// ------------------------------------------------------------------------------------------------
// fused ring flash-attention backward: two kernels, no atomics, no cross-rank reduction.
//   dq kernel   : Q-stationary  (like forward), streams K/V tiles of every visible owner
//   dkdv kernel : KV-stationary, streams Q / dO / lse / delta tiles of every rank that can see the keys
// Both address kv_buf [world][2][b*hk][n_k][d] and qdo_buf [world][2][b*h][n_q][d] (16 bit) plus stat_buf
// [world][2][b*h][n_pad] (fp32: lse*log2e, delta) by owner slot.  Gather mode: slot `rank` is written
// locally, the other slots arrive over NVLink (copy engines on a side stream, or an earlier kernel) and
// are published through the per-owner ready flags.  Hop mode (memory = "ring"): one launch per ring hop,
// every buffer is one owner's slot (its base shifted so that the owner's slot index lands on it), and the
// fp32 accumulators travel between the launches in `carry`.
// ------------------------------------------------------------------------------------------------
struct AttnBwdParams : AttnProblem {
  int n_pad;
  const float* stat;           // [world][2][b*h][n_pad]
  void* dq;                    // [b, n_q, h, d]
  void* dk;                    // [b, n_k, hk, d]
  void* dv;                    // [b, n_k, hk, d]
  const uint32_t* ready;       // [world] flags: slot o usable once ready[o] >= ready_target (may be null)
  uint32_t ready_target;
  // hop-at-a-time mode: dq kernel fp32 [b, n_q, h, d]; dkdv kernel fp32 [2][b, n_k, hk, d] (dK, dV); both unscaled
  float* carry;
  int carry_in;   // 1: every item's accumulator starts from `carry` instead of zero
  int carry_out;  // 1: store the fp32 accumulator to `carry` instead of the scaled 16-bit output
};

template <int D>
void launch_attn_bwd_dq(const CUtensorMap& map_qd, const CUtensorMap& map_kv, const AttnBwdParams& p, int num_sms,
                        cudaStream_t stream);
template <int D>
void launch_attn_bwd_dkdv(const CUtensorMap& map_qd64, const CUtensorMap& map_kv, const AttnBwdParams& p,
                          int num_sms, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// one-kernel (5-GEMM) ring backward, head dim 128 (attn_bwd_fused_sm100.cu)
//   local  : qdo [2][b*h][n_q][d] 16 bit, stat [2][b*h][n_pad] fp32 (lse*log2e, delta), dq_acc fp32 [b*h][n_pad][d]
//   K/V    : gather buffer [world][2][b*hk][n_k][d]; slot o usable once ready[o] >= ready_target (null: always)
//   dK/dV  : ring_reduce == 0: 16 bit [b, n_k, hk, d] written directly (single rank)
//            ring_reduce == 1: added into owner o's fp32 [2][b*hk][nk_pad][d] accumulator through map_dkv[o]
// ------------------------------------------------------------------------------------------------
struct AttnBwdFusedParams : AttnProblem {
  int n_pad, nk_pad;
  int self_owner[1];         // = {rank}: the streamed queries are always local
  const float* stat;
  const uint32_t* ready;
  uint32_t ready_target;
  void* dk;
  void* dv;
  int ring_reduce;
  alignas(64) CUtensorMap map_dkv[kMaxWorld];
};
void launch_attn_bwd_fused(const CUtensorMap& map_qd64, const CUtensorMap& map_kv, const CUtensorMap& map_dq,
                           const AttnBwdFusedParams& p, int num_sms, cudaStream_t stream);
size_t attn_bwd_fused_smem_bytes();
// fp32 accumulator [b*h][n_pad][d] -> 16 bit [b][n][h][d], multiplied by scale
void launch_acc_convert(const float* acc, void* out, int batch, int heads, int n, int n_pad, int d, float scale,
                        int is_bf16, cudaStream_t stream);

// q, o, do: [b, n, h, d] contiguous 16 bit; lse: [b, h, n] fp32 (natural log).
// Writes this rank's slot: qdo_slot [2][b*h][n][d] (q, do) and stat_slot [2][b*h][n_pad] (lse*log2e, delta).
void launch_bwd_prep(const void* q, const void* o, const void* dout, const float* lse, void* qdo_slot,
                     float* stat_slot, int batch, int n, int heads, int d, int n_pad, int is_bf16,
                     cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// tree-attention decode (tree_decode_sm100.cu): ONE persistent cooperative kernel per rank and step
// ------------------------------------------------------------------------------------------------
struct TreeDecodeParams {
  const void* q;            // [b, h, d]; q_kind 0 bf16, 1 fp16, 2 fp32
  int q_kind;
  const void* k;            // [b*hk, n, d]; kv_kind 0 bf16, 1 fp16, 2 fp8-e4m3
  const void* v;
  int kv_kind;
  const float* k_scale;     // null or [b*hk][n_scale_blocks] fp32: one scale per `scale_block` keys (multiple of 64)
  const float* v_scale;
  int scale_block, n_scale_blocks;
  int batch, heads, kv_heads, n, splits;
  float scale_log2;         // softmax scale * log2(e)
  float* scratch;           // [b*hk][splits][g][d+4] fp32 (used when splits > 1)
  uint32_t* group_done;     // [b*hk*ceil(g/4)] zero-initialised, self-resetting
  uint32_t* counters;       // [4] zero-initialised: queue head, grid-barrier count, grid-barrier generation, epoch
  // cross-rank merge.  Row = (out[d], lse*log2e, valid, 0, 0); buffers hold TWO halves (alternating calls).
  int world, rank;
  float* partial_local;               // this rank's [2][b*h][d+4]
  const float* partials[kMaxWorld];   // every rank's buffer (peer-mapped), index = rank
  float* aux_local;                   // this rank's [2][2][b*h] (NVLS path: ordered-int lse, weights)
  uint32_t* pads[kMaxWorld];          // signal pads: pads[r] lives on rank r, [2 rounds][kMaxWorld] words
  const float* mc_partial;            // multicast (NVLS) mapping of the partial buffers, null -> P2P loads
  const float* mc_aux;                // multicast mapping of the aux buffers
  void* out;                          // [b*h][d]; out_kind 0 fp16, 1 bf16, 2 fp32
  int out_kind;
  float eps;
};
int tree_decode_max_ctas(int d, int kv_kind, int num_sms);
void launch_tree_decode(const TreeDecodeParams& p, int d, int grid, cudaStream_t stream);
// tcgen05 variant (tree_decode_tc_sm100.cu): head dim 128; map_k / map_v: K, V as (d, n, b*hk) with a 128-byte x 128-key box
int tree_decode_tc_max_ctas(int kv_kind, int num_sms);
void launch_tree_decode_tc(const CUtensorMap& map_k, const CUtensorMap& map_v, const TreeDecodeParams& p, int grid,
                           cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// misc kernels (elementwise_sm100.cu)
// ------------------------------------------------------------------------------------------------
// k, v [b, n, hk, d] (arbitrary batch/seq/head strides, unit d stride) -> slot [2][b*hk][n][d]
// which: bit 0 = pack the K half, bit 1 = pack the V half
void launch_pack_kv(const void* k, const void* v, void* slot, int batch, int n, int kv_heads, int d,
                    long long k_sb, long long k_sn, long long k_sh, long long v_sb, long long v_sn,
                    long long v_sh, int which, cudaStream_t stream);

// rotary embedding (rotate-half convention) fused with a layout change; see elementwise_sm100.cu:rotary_kernel
void launch_rotary(const void* x, void* out, const float* angles, int astride, int batch, int n, int heads, int d,
                   long long sb, long long sn, long long sh, long long ob, long long on, long long oh, float sign,
                   int is_bf16, cudaStream_t stream);

// cross-device barrier on symmetric signal pads: every rank bumps its epoch slot on every peer and
// waits until all peers have bumped its own pad.
struct BarrierParams {
  int world;
  int rank;
  uint32_t epoch;
  uint32_t* pads[kMaxWorld];  // pads[r] = signal pad living on rank r (peer-mapped), kMaxWorld words each
};
void launch_device_barrier(const BarrierParams& p, cudaStream_t stream);

}  // namespace rab
