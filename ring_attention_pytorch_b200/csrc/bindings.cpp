// torch.ops.rab.* bindings.  Only this file sees torch headers.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/torch.h>

#include <vector>

#include "kernels.h"
#include "symm.h"

namespace {

using torch::Tensor;

int sm_count() {
  static int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v;
  }();
  return n;
}

// bench.py hook: when set, the next forward launches record the activity window of their in-kernel K/V fetchers
unsigned long long* g_fetch_times = nullptr;
int64_t g_fetch_times_rows = 0;

void set_fetch_timing(const c10::optional<Tensor>& t) {
  if (!t.has_value()) {
    g_fetch_times = nullptr;
    g_fetch_times_rows = 0;
    return;
  }
  TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kLong && t->is_contiguous() && t->dim() == 2 && t->size(1) == 2);
  g_fetch_times = reinterpret_cast<unsigned long long*>(t->data_ptr<int64_t>());
  g_fetch_times_rows = t->size(0);
}

void check_16bit(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kBFloat16 || t.scalar_type() == at::kHalf, name, " must be bf16 or fp16");
}

// ---------------------------------------------------------------------------------------------
// descriptor probe
// ---------------------------------------------------------------------------------------------
Tensor umma_probe(const Tensor& a, const Tensor& b, int64_t mode, int64_t n, int64_t k, int64_t idesc,
                  int64_t a_lbo, int64_t a_sbo, int64_t b_lbo, int64_t b_sbo, int64_t b_kstep) {
  check_16bit(a, "a");
  check_16bit(b, "b");
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous());
  c10::cuda::CUDAGuard guard(a.device());
  CUtensorMap map_a, map_b;
  if (mode == 3) {  // a is At [k, 128] (MN-major A); b [k, 64] is written to shared memory by the kernel's threads
    TORCH_CHECK(a.size(0) == k && a.size(1) == 128 && b.size(0) == k && b.size(1) == 64 && n == 64);
    uint64_t adims[2] = {128, (uint64_t)k};
    uint64_t astr[1] = {128 * 2};
    uint32_t abox[2] = {64, (uint32_t)k};
    map_a = rab::make_tmap_bf16(a.data_ptr(), 2, adims, astr, abox, rab::TmapSwizzle::B128);
    map_b = map_a;
  } else {
    TORCH_CHECK(a.size(0) == 128 && a.size(1) == k);
    uint64_t adims[2] = {(uint64_t)k, 128};
    uint64_t astr[1] = {(uint64_t)k * 2};
    uint32_t abox[2] = {64, 128};
    map_a = rab::make_tmap_bf16(a.data_ptr(), 2, adims, astr, abox, rab::TmapSwizzle::B128);
  }
  if (mode == 3) {
  } else if (mode == 0) {
    TORCH_CHECK(b.size(0) == n && b.size(1) == k);
    uint64_t bdims[2] = {(uint64_t)k, (uint64_t)n};
    uint64_t bstr[1] = {(uint64_t)k * 2};
    uint32_t bbox[2] = {64, (uint32_t)n};
    map_b = rab::make_tmap_bf16(b.data_ptr(), 2, bdims, bstr, bbox, rab::TmapSwizzle::B128);
  } else {
    TORCH_CHECK(b.size(0) == k && b.size(1) == n);
    uint64_t bdims[2] = {(uint64_t)n, (uint64_t)k};
    uint64_t bstr[1] = {(uint64_t)n * 2};
    uint32_t bbox[2] = {64, (uint32_t)k};
    map_b = rab::make_tmap_bf16(b.data_ptr(), 2, bdims, bstr, bbox, rab::TmapSwizzle::B128);
  }
  rab::ProbeParams p;
  p.mode = (int)mode;
  p.n = (int)n;
  p.k = (int)k;
  p.idesc = (uint32_t)idesc;
  p.a_lbo = (uint32_t)a_lbo;
  p.a_sbo = (uint32_t)a_sbo;
  p.b_lbo = (uint32_t)b_lbo;
  p.b_sbo = (uint32_t)b_sbo;
  p.b_kstep_bytes = (uint32_t)b_kstep;
  Tensor out = torch::empty({128, n}, a.options().dtype(at::kFloat));
  rab::launch_umma_probe(map_a, map_b, p, mode == 3 ? b.data_ptr() : a.data_ptr(), out.data_ptr<float>(),
                         at::cuda::getCurrentCUDAStream());
  return out;
}

// cycles for `reps` back-to-back tcgen05.mma of one flavour on `ctas` SMs: returns [ctas, 2] (total, issue-side)
Tensor umma_rate(int64_t mode, int64_t n, int64_t reps, int64_t alt, int64_t ctas) {
  TORCH_CHECK(n == 64 || n == 128 || n == 256, "n must be 64, 128 or 256");
  Tensor out = torch::zeros({ctas, 2}, torch::dtype(at::kLong).device(at::kCUDA));
  rab::launch_umma_rate((int)mode, (int)n, (int)reps, (int)alt, (int)ctas,
                        reinterpret_cast<long long*>(out.data_ptr<int64_t>()), at::cuda::getCurrentCUDAStream());
  return out;
}

// ---------------------------------------------------------------------------------------------
// the attention problem: every attention op ends with these arguments, in this order
// (ops/fused.py:AttnProblem.tail produces them)
// ---------------------------------------------------------------------------------------------
#define PROBLEM_SCHEMA                                                                                               \
  "Tensor? kmask_bits, int batch, int heads, int kv_heads, int rank, bool causal, int window, float scale, float " \
  "softclamp, int pos_stride, int seg_len, int[] base0, int[] base1, int q_pos_offset, int[] hop_owner"
#define PROBLEM_PARAMS                                                                                               \
  const c10::optional<Tensor>& kmask_bits, int64_t batch, int64_t heads, int64_t kv_heads, int64_t rank, bool causal, \
      int64_t window, double scale, double softclamp, int64_t pos_stride, int64_t seg_len, at::IntArrayRef base0,  \
      at::IntArrayRef base1, int64_t q_pos_offset, at::IntArrayRef hop_owner
#define PROBLEM_ARGS                                                                                              \
  kmask_bits, batch, heads, kv_heads, rank, causal, window, scale, softclamp, pos_stride, seg_len, base0, base1, \
      q_pos_offset, hop_owner

// Fills `p` from the problem arguments and the K/V buffer kv_buf [slots][2][b*hk][n_k][d] (16 bit).  The ring size is
// the length of the position map.  The buffer holds either every owner's slot, and then hop 0 is this rank, or one
// owner's slot only (memory = "ring": one launch per hop), and then the launch visits exactly that owner.
void parse_problem(rab::AttnProblem& p, const Tensor& kv_buf, int n_q, PROBLEM_PARAMS) {
  check_16bit(kv_buf, "kv_buf");
  TORCH_CHECK(kv_buf.dim() == 5 && kv_buf.is_contiguous(), "kv_buf must be contiguous [slots, 2, b*hk, n_k, d]");
  TORCH_CHECK(kv_buf.size(1) == 2 && kv_buf.size(2) == batch * kv_heads);
  TORCH_CHECK(kv_buf.size(4) == 64 || kv_buf.size(4) == 128, "head dim must be 64 or 128");
  TORCH_CHECK(heads % kv_heads == 0);
  const int world = (int)base0.size(), slots = (int)kv_buf.size(0);
  TORCH_CHECK(world >= 1 && world <= rab::kMaxWorld && (int)base1.size() == world,
              "position map needs one base per rank, at most ", rab::kMaxWorld);
  TORCH_CHECK(rank >= 0 && rank < world);
  TORCH_CHECK(hop_owner.size() >= 1 && (int)hop_owner.size() <= world);
  for (int64_t o : hop_owner) TORCH_CHECK(o >= 0 && o < world, "hop owner out of range");
  if (slots == world) {
    TORCH_CHECK(hop_owner[0] == rank, "hop 0 must be this rank");
  } else {
    TORCH_CHECK(slots == 1 && hop_owner.size() == 1, "a one-slot K/V buffer serves exactly one hop");
  }
  p.batch = (int)batch; p.heads = (int)heads; p.kv_heads = (int)kv_heads;
  p.n_q = n_q; p.n_k = (int)kv_buf.size(3);
  p.world = world; p.rank = (int)rank;
  p.causal = causal; p.window = (int)window;
  p.is_bf16 = kv_buf.scalar_type() == at::kBFloat16;
  p.scale = (float)scale; p.softclamp = (float)softclamp;
  p.pos.stride = (int)pos_stride;
  p.pos.seg_len = (int)seg_len;
  for (int i = 0; i < world; ++i) {
    p.pos.base0[i] = (int)base0[i];
    p.pos.base1[i] = (int)base1[i];
  }
  p.q_pos_offset = (int)q_pos_offset;
  p.hop_count = (int)hop_owner.size();
  for (int i = 0; i < p.hop_count; ++i) p.hop_owner[i] = (int)hop_owner[i];
  if (kmask_bits.has_value()) {
    const Tensor& km = *kmask_bits;
    TORCH_CHECK(km.is_cuda() && km.scalar_type() == at::kInt && km.is_contiguous() && km.dim() == 3);
    TORCH_CHECK(km.size(0) == world && km.size(1) == batch && km.size(2) % 4 == 0 && km.size(2) * 32 >= p.n_k);
    p.kmask_bits = reinterpret_cast<const uint32_t*>(km.data_ptr<int>());
    p.kmask_words = km.size(2);
  }
}

// Address of owner slot 0 of a per-owner buffer [slots][...] as the kernels see it.  They address owner o's data at
// slot o: a buffer with every owner's slot is used as it is, and a one-slot buffer IS the slot of `owner`, so its base
// moves down by that many slots (only that slot is ever dereferenced).
uint8_t* slot0(const Tensor& buf, int world, int owner) {
  const size_t slot_bytes = buf.nbytes() / buf.size(0);
  const int shift = buf.size(0) == world ? 0 : owner;
  return reinterpret_cast<uint8_t*>(buf.data_ptr()) - shift * slot_bytes;
}

// K/V of every owner, [world][2][b*hk][n_k][d] -> dims (d, n_k, b*hk, 2*world), box (64, 128, 1, 1); a one-slot
// kv_buf is the slot of `owner`
CUtensorMap make_kv_map(const Tensor& kv_buf, const rab::AttnProblem& p, int owner) {
  const uint64_t d = kv_buf.size(4), rows = (uint64_t)p.batch * p.kv_heads;
  uint64_t dims[4] = {d, (uint64_t)p.n_k, rows, (uint64_t)2 * p.world};
  uint64_t str[3] = {d * 2, (uint64_t)p.n_k * d * 2, rows * p.n_k * d * 2};
  uint32_t box[4] = {64, 128, 1, 1};
  return rab::make_tmap_bf16(slot0(kv_buf, p.world, owner), 4, dims, str, box, rab::TmapSwizzle::B128);
}

// per-owner ready flags: int32, one per ring rank (null when not given)
uint32_t* ready_flags(const c10::optional<Tensor>& ready, int world) {
  if (!ready.has_value()) return nullptr;
  TORCH_CHECK(ready->is_cuda() && ready->scalar_type() == at::kInt && ready->numel() >= world,
              "ready must be int32 [world] on the GPU");
  return reinterpret_cast<uint32_t*>(ready->data_ptr<int>());
}

// ---------------------------------------------------------------------------------------------
// fused ring attention forward
// ---------------------------------------------------------------------------------------------
void parse_fwd(rab::AttnFwdParams& p, const Tensor& q, const Tensor& kv_buf, PROBLEM_PARAMS) {
  check_16bit(q, "q");
  TORCH_CHECK(q.dim() == 4 && q.is_contiguous(), "q must be contiguous [b, n, h, d]");
  std::memset(&p, 0, sizeof(p));
  parse_problem(p, kv_buf, (int)q.size(1), PROBLEM_ARGS);
  TORCH_CHECK(kv_buf.scalar_type() == q.scalar_type());
  TORCH_CHECK(q.size(0) == batch && q.size(2) == heads && q.size(3) == kv_buf.size(4));
  p.slot_bytes = kv_buf.nbytes() / kv_buf.size(0);
  p.kv_local = slot0(kv_buf, p.world, p.hop_owner[0]);
}

std::tuple<Tensor, Tensor> launch_fwd(const Tensor& q, const Tensor& kv_buf, rab::AttnFwdParams& p) {
  c10::cuda::CUDAGuard guard(q.device());
  const int b = p.batch, n_q = p.n_q, h = p.heads, d = q.size(3);
  Tensor o = torch::empty_like(q);
  Tensor lse = torch::empty({b, h, n_q}, q.options().dtype(at::kFloat));
  p.o = o.data_ptr();
  p.lse = lse.data_ptr<float>();
  // Q: [b, n, h, d] -> dims (d, h, n, b), box (64, 1, 128, 1)
  uint64_t qdims[4] = {(uint64_t)d, (uint64_t)h, (uint64_t)n_q, (uint64_t)b};
  uint64_t qstr[3] = {(uint64_t)d * 2, (uint64_t)h * d * 2, (uint64_t)n_q * h * d * 2};
  uint32_t qbox[4] = {64, 1, 128, 1};
  CUtensorMap map_q = rab::make_tmap_bf16(q.data_ptr(), 4, qdims, qstr, qbox, rab::TmapSwizzle::B128);
  CUtensorMap map_kv = make_kv_map(kv_buf, p, p.hop_owner[0]);
  auto stream = at::cuda::getCurrentCUDAStream();
  if (d == 128) {
    rab::launch_attn_fwd<128>(map_q, map_kv, p, sm_count(), stream);
  } else {
    rab::launch_attn_fwd<64>(map_q, map_kv, p, sm_count(), stream);
  }
  return {o, lse};
}

// The whole ring in one launch: kv_buf [world, 2, b*hk, n_k, d] holds this rank's slot; the kernel's fetchers pull
// owner o's slot from peer_ptrs[o] (0: already local) and publish it through the ready flags.
std::tuple<Tensor, Tensor> attn_fwd(const Tensor& q, const Tensor& kv_buf, at::IntArrayRef peer_ptrs,
                                    const Tensor& ready, PROBLEM_PARAMS) {
  rab::AttnFwdParams p;
  parse_fwd(p, q, kv_buf, PROBLEM_ARGS);
  TORCH_CHECK(kv_buf.size(0) == p.world && (int)peer_ptrs.size() == p.world, "attn_fwd needs every owner's slot");
  for (int i = 0; i < p.world; ++i)
    p.kv_peer[i] = peer_ptrs[i] ? reinterpret_cast<const uint8_t*>(peer_ptrs[i]) : p.kv_local + i * p.slot_bytes;
  p.ready = ready_flags(ready, p.world);
  c10::cuda::CUDAGuard guard(q.device());
  rab::cuda_check(cudaMemsetAsync(p.ready, 0, sizeof(uint32_t) * p.world, at::cuda::getCurrentCUDAStream()),
                  "ready memset");
  p.fetch_times = (g_fetch_times != nullptr && g_fetch_times_rows >= sm_count()) ? g_fetch_times : nullptr;
  return launch_fwd(q, kv_buf, p);
}

// One ring hop of the forward: q against the one owner slot kv_slot [1, 2, b*hk, n_k, d] of owner hop_owner[0].
// carry_o fp32 [b, n_q, h, d] and carry_ml fp32 [2, b*h, n_q] hold the online-softmax state between hops; the launch
// with carry_out = false writes the final O / lse.
std::tuple<Tensor, Tensor> attn_fwd_hop(const Tensor& q, const Tensor& kv_slot, Tensor carry_o, Tensor carry_ml,
                                        bool carry_in, bool carry_out, PROBLEM_PARAMS) {
  rab::AttnFwdParams p;
  parse_fwd(p, q, kv_slot, PROBLEM_ARGS);
  TORCH_CHECK(kv_slot.size(0) == 1, "attn_fwd_hop takes one owner's slot");
  const int64_t b = p.batch, n_q = p.n_q, h = p.heads, d = q.size(3);
  TORCH_CHECK(carry_o.is_cuda() && carry_o.scalar_type() == at::kFloat && carry_o.is_contiguous() &&
              carry_o.numel() == b * n_q * h * d, "carry_o must be fp32 [b, n_q, h, d]");
  TORCH_CHECK(carry_ml.is_cuda() && carry_ml.scalar_type() == at::kFloat && carry_ml.is_contiguous() &&
              carry_ml.numel() == 2 * b * h * n_q, "carry_ml must be fp32 [2, b*h, n_q]");
  p.all_ready = 1;
  p.carry_o = carry_o.data_ptr<float>();
  p.carry_ml = carry_ml.data_ptr<float>();
  p.carry_in = carry_in;
  p.carry_out = carry_out;
  return launch_fwd(q, kv_slot, p);
}

// ---------------------------------------------------------------------------------------------
// fused ring attention backward
// ---------------------------------------------------------------------------------------------
void bwd_prep(const Tensor& q, const Tensor& o, const Tensor& dout, const Tensor& lse, Tensor qdo_buf,
              Tensor stat_buf, int64_t rank) {
  check_16bit(q, "q");
  TORCH_CHECK(q.is_contiguous() && o.is_contiguous() && dout.is_contiguous() && lse.is_contiguous());
  TORCH_CHECK(o.scalar_type() == q.scalar_type() && dout.scalar_type() == q.scalar_type());
  TORCH_CHECK(lse.scalar_type() == at::kFloat && stat_buf.scalar_type() == at::kFloat);
  const int b = q.size(0), n = q.size(1), h = q.size(2), d = q.size(3);
  TORCH_CHECK(qdo_buf.dim() == 5 && qdo_buf.is_contiguous() && qdo_buf.size(1) == 2 && qdo_buf.size(2) == b * h &&
              qdo_buf.size(3) == n && qdo_buf.size(4) == d && qdo_buf.scalar_type() == q.scalar_type());
  TORCH_CHECK(stat_buf.dim() == 4 && stat_buf.is_contiguous() && stat_buf.size(1) == 2 && stat_buf.size(2) == b * h);
  const int n_pad = stat_buf.size(3);
  TORCH_CHECK(n_pad >= n && n_pad % 64 == 0);
  c10::cuda::CUDAGuard guard(q.device());
  rab::launch_bwd_prep(q.data_ptr(), o.data_ptr(), dout.data_ptr(), lse.data_ptr<float>(),
                       qdo_buf[rank].data_ptr(), stat_buf[rank].data_ptr<float>(), b, n, h, d, n_pad,
                       q.scalar_type() == at::kBFloat16, at::cuda::getCurrentCUDAStream());
}

struct BwdSetup {
  rab::AttnBwdParams p;
  CUtensorMap map_qd128, map_qd64, map_kv;
};

// The two-kernel backward's buffers: qdo_buf [slots][2][b*h][n_q][d], kv_buf [slots][2][b*hk][n_k][d], stat_buf
// [slots][2][b*h][n_pad].  Each holds every owner's slot (gathered, slots = world) or the one slot of qdo_owner /
// kv_owner (the Q/dO buffer and the statistics share their owner).
BwdSetup make_bwd_setup(const Tensor& qdo_buf, const Tensor& kv_buf, const Tensor& stat_buf, bool one_slot,
                        bool kv_is_own, PROBLEM_PARAMS) {
  check_16bit(qdo_buf, "qdo_buf");
  TORCH_CHECK(qdo_buf.is_contiguous() && stat_buf.is_contiguous());
  TORCH_CHECK(qdo_buf.dim() == 5 && stat_buf.dim() == 4);
  BwdSetup s;
  rab::AttnBwdParams& p = s.p;
  std::memset(&p, 0, sizeof(p));
  parse_problem(p, kv_buf, (int)qdo_buf.size(3), PROBLEM_ARGS);
  const int world = p.world, n_q = p.n_q, d = kv_buf.size(4);
  const int slots = one_slot ? 1 : world;
  TORCH_CHECK(kv_buf.size(0) == slots, one_slot ? "one owner's K/V slot expected" :
              "the two-kernel backward needs every owner's slot");
  TORCH_CHECK(qdo_buf.scalar_type() == kv_buf.scalar_type(), "qdo_buf and kv_buf must share a dtype");
  TORCH_CHECK(qdo_buf.size(0) == slots && qdo_buf.size(1) == 2 && qdo_buf.size(2) == batch * heads &&
              qdo_buf.size(4) == d, "qdo_buf must be [slots, 2, b*h, n_q, d]");
  TORCH_CHECK(stat_buf.size(0) == slots && stat_buf.size(1) == 2 && stat_buf.size(2) == batch * heads,
              "stat_buf must be [slots, 2, b*h, n_pad]");
  if (one_slot) {
    TORCH_CHECK(stat_buf.scalar_type() == at::kFloat && stat_buf.size(3) % 64 == 0 && stat_buf.size(3) >= n_q,
                "stat_buf must be fp32 with n_pad >= n_q, n_pad % 64 == 0");
  }
  // the dQ kernel reads this rank's queries against the hop owner's keys, the dK/dV kernel this rank's keys against
  // the hop owner's queries
  const int kv_owner = kv_is_own ? p.rank : p.hop_owner[0];
  const int q_owner = kv_is_own ? p.hop_owner[0] : p.rank;
  p.n_pad = stat_buf.size(3);
  p.stat = reinterpret_cast<const float*>(slot0(stat_buf, world, q_owner));
  uint64_t qdims[4] = {(uint64_t)d, (uint64_t)n_q, (uint64_t)batch * heads, (uint64_t)2 * world};
  uint64_t qstr[3] = {(uint64_t)d * 2, (uint64_t)n_q * d * 2, (uint64_t)batch * heads * n_q * d * 2};
  uint32_t qbox128[4] = {64, 128, 1, 1};
  uint32_t qbox64[4] = {64, 64, 1, 1};
  uint8_t* qd0 = slot0(qdo_buf, world, q_owner);
  s.map_qd128 = rab::make_tmap_bf16(qd0, 4, qdims, qstr, qbox128, rab::TmapSwizzle::B128);
  s.map_qd64 = rab::make_tmap_bf16(qd0, 4, qdims, qstr, qbox64, rab::TmapSwizzle::B128);
  s.map_kv = make_kv_map(kv_buf, p, kv_owner);
  return s;
}

// gathered buffers: slot o usable once ready[o] >= ready_target (no flags: all usable)
BwdSetup make_bwd_gather_setup(const Tensor& qdo_buf, const Tensor& kv_buf, const Tensor& stat_buf,
                               const c10::optional<Tensor>& ready, int64_t ready_target, PROBLEM_PARAMS) {
  BwdSetup s = make_bwd_setup(qdo_buf, kv_buf, stat_buf, false, false, PROBLEM_ARGS);
  s.p.ready = ready_flags(ready, s.p.world);
  s.p.ready_target = s.p.ready ? (uint32_t)ready_target : 0;
  return s;
}

// one ring hop: `carry` holds the fp32 accumulators between the launches (see AttnBwdParams); unused, and then
// unchecked, when neither flag is set
void set_bwd_carry(rab::AttnBwdParams& p, Tensor& carry, at::IntArrayRef shape, bool carry_in, bool carry_out,
                   const char* what) {
  if (!carry_in && !carry_out) return;
  TORCH_CHECK(carry.is_cuda() && carry.scalar_type() == at::kFloat && carry.is_contiguous() && carry.sizes() == shape,
              "carry must be contiguous fp32 ", what, " ", shape);
  p.carry = carry.data_ptr<float>();
  p.carry_in = carry_in;
  p.carry_out = carry_out;
}

// dQ [b, n_q, h, d] 16 bit, or (carry_out) an empty tensor: the accumulator stays in the carry
Tensor launch_bwd_dq(BwdSetup& s, const Tensor& kv_buf, int64_t batch, int64_t heads) {
  const int d = kv_buf.size(4);
  Tensor dq = torch::empty({s.p.carry_out ? 0 : batch, s.p.n_q, heads, d}, kv_buf.options());
  s.p.dq = s.p.carry_out ? nullptr : dq.data_ptr();
  auto stream = at::cuda::getCurrentCUDAStream();
  if (d == 128) {
    rab::launch_attn_bwd_dq<128>(s.map_qd128, s.map_kv, s.p, sm_count(), stream);
  } else {
    rab::launch_attn_bwd_dq<64>(s.map_qd128, s.map_kv, s.p, sm_count(), stream);
  }
  return dq;
}

// dK, dV [b, n_k, hk, d] 16 bit, or (carry_out) empty tensors: the accumulators stay in the carry
std::tuple<Tensor, Tensor> launch_bwd_dkdv(BwdSetup& s, const Tensor& kv_buf, int64_t batch, int64_t kv_heads) {
  const int d = kv_buf.size(4);
  Tensor dk = torch::empty({s.p.carry_out ? 0 : batch, s.p.n_k, kv_heads, d}, kv_buf.options());
  Tensor dv = torch::empty({s.p.carry_out ? 0 : batch, s.p.n_k, kv_heads, d}, kv_buf.options());
  s.p.dk = s.p.carry_out ? nullptr : dk.data_ptr();
  s.p.dv = s.p.carry_out ? nullptr : dv.data_ptr();
  auto stream = at::cuda::getCurrentCUDAStream();
  if (d == 128) {
    rab::launch_attn_bwd_dkdv<128>(s.map_qd64, s.map_kv, s.p, sm_count(), stream);
  } else {
    rab::launch_attn_bwd_dkdv<64>(s.map_qd64, s.map_kv, s.p, sm_count(), stream);
  }
  return {dk, dv};
}

Tensor attn_bwd_dq(const Tensor& qdo_buf, const Tensor& kv_buf, const Tensor& stat_buf,
                   const c10::optional<Tensor>& ready, int64_t ready_target, PROBLEM_PARAMS) {
  c10::cuda::CUDAGuard guard(kv_buf.device());
  BwdSetup s = make_bwd_gather_setup(qdo_buf, kv_buf, stat_buf, ready, ready_target, PROBLEM_ARGS);
  return launch_bwd_dq(s, kv_buf, batch, heads);
}

// One ring hop of the dQ kernel: this rank's qdo_own [1, 2, b*h, n_q, d] / stat_own [1, 2, b*h, n_pad] against the
// one K/V slot kv_slot [1, 2, b*hk, n_k, d] of owner hop_owner[0].  carry fp32 [b, n_q, h, d] (unscaled dQ) travels
// between the launches; with carry_out the result stays in it and an empty tensor is returned.
Tensor attn_bwd_dq_hop(const Tensor& qdo_own, const Tensor& kv_slot, const Tensor& stat_own, Tensor carry,
                       bool carry_in, bool carry_out, PROBLEM_PARAMS) {
  c10::cuda::CUDAGuard guard(kv_slot.device());
  BwdSetup s = make_bwd_setup(qdo_own, kv_slot, stat_own, true, false, PROBLEM_ARGS);
  set_bwd_carry(s.p, carry, {batch, s.p.n_q, heads, kv_slot.size(4)}, carry_in, carry_out, "[b, n_q, h, d]");
  return launch_bwd_dq(s, kv_slot, batch, heads);
}

std::tuple<Tensor, Tensor> attn_bwd_dkdv(const Tensor& qdo_buf, const Tensor& kv_buf, const Tensor& stat_buf,
                                         const c10::optional<Tensor>& ready, int64_t ready_target, PROBLEM_PARAMS) {
  c10::cuda::CUDAGuard guard(kv_buf.device());
  BwdSetup s = make_bwd_gather_setup(qdo_buf, kv_buf, stat_buf, ready, ready_target, PROBLEM_ARGS);
  return launch_bwd_dkdv(s, kv_buf, batch, kv_heads);
}

// One ring hop of the dK/dV kernel: this rank's kv_own [1, 2, b*hk, n_k, d] against the one Q/dO slot qdo_slot
// [1, 2, b*h, n_q, d] / stat_slot [1, 2, b*h, n_pad] of query owner hop_owner[0].  carry fp32 [2, b, n_k, hk, d]
// (unscaled dK, dV) travels between the launches; with carry_out the result stays in it and empty tensors are returned.
std::tuple<Tensor, Tensor> attn_bwd_dkdv_hop(const Tensor& qdo_slot, const Tensor& kv_own, const Tensor& stat_slot,
                                             Tensor carry, bool carry_in, bool carry_out, PROBLEM_PARAMS) {
  c10::cuda::CUDAGuard guard(kv_own.device());
  BwdSetup s = make_bwd_setup(qdo_slot, kv_own, stat_slot, true, true, PROBLEM_ARGS);
  set_bwd_carry(s.p, carry, {2, batch, s.p.n_k, kv_heads, kv_own.size(4)}, carry_in, carry_out,
                "[2, b, n_k, hk, d]");
  return launch_bwd_dkdv(s, kv_own, batch, kv_heads);
}

// One-kernel (5-GEMM) ring backward, head dim 128 (attn_bwd_fused_sm100.cu).
//   qdo [2][b*h][n_q][d] 16 bit and stat [2][b*h][n_pad] fp32: this rank's bwd_prep output
//   kv_buf: the K/V gather [world][2][b*hk][n_k][d] (slot o valid once ready[o] >= ready_target; no flags: all valid),
//           or one owner's slot [1][2][b*hk][n_k][d] (memory = "ring": one launch per hop)
//   dq_acc fp32 [b*h][n_pad][d], zeroed by the caller: dQ (unscaled) is ADDED into it
//   dkv_acc_ptrs: empty -> dK, dV are returned as 16 bit [b, n_k, hk, d] (single rank);
//                 else one pointer per ring rank to that rank's zeroed fp32 [2][b*hk][nk_pad][d] accumulator (peer
//                 mapped): the kernel adds its dK / dV tiles into the owner's accumulator and returns empty tensors.
// dq_acc and the dK / dV accumulators keep adding up across the per-hop launches.
std::tuple<Tensor, Tensor> attn_bwd_ring(const Tensor& qdo, const Tensor& kv_buf, const Tensor& stat, Tensor dq_acc,
                                         const c10::optional<Tensor>& ready, int64_t ready_target,
                                         at::IntArrayRef dkv_acc_ptrs, int64_t nk_pad, PROBLEM_PARAMS) {
  check_16bit(qdo, "qdo");
  TORCH_CHECK(qdo.is_contiguous() && stat.is_contiguous() && dq_acc.is_contiguous());
  TORCH_CHECK(qdo.dim() == 4 && stat.dim() == 3 && dq_acc.dim() == 3);
  rab::AttnBwdFusedParams p;
  std::memset(&p, 0, sizeof(p));
  parse_problem(p, kv_buf, (int)qdo.size(2), PROBLEM_ARGS);
  const int world = p.world, n_q = p.n_q, n_k = p.n_k, n_pad = stat.size(2), d = kv_buf.size(4);
  TORCH_CHECK(d == 128, "attn_bwd_ring: head dim 128 only");
  TORCH_CHECK(qdo.size(0) == 2 && qdo.size(1) == batch * heads && qdo.size(3) == d);
  TORCH_CHECK(stat.size(0) == 2 && stat.size(1) == batch * heads && stat.scalar_type() == at::kFloat);
  TORCH_CHECK(n_pad % 64 == 0 && n_pad >= n_q);
  TORCH_CHECK(dq_acc.scalar_type() == at::kFloat && dq_acc.size(0) == batch * heads && dq_acc.size(1) == n_pad &&
              dq_acc.size(2) == d);
  c10::cuda::CUDAGuard guard(kv_buf.device());
  auto stream = at::cuda::getCurrentCUDAStream();

  p.n_pad = n_pad; p.nk_pad = (int)nk_pad;
  p.self_owner[0] = (int)rank;
  p.stat = stat.data_ptr<float>();
  p.ready = ready_flags(ready, world);
  p.ready_target = p.ready ? (uint32_t)ready_target : 0;
  // local Q / dO: dims (d, n_q, b*h, 2), box (64, 64, 1, 1)
  uint64_t qdims[4] = {(uint64_t)d, (uint64_t)n_q, (uint64_t)batch * heads, 2};
  uint64_t qstr[3] = {(uint64_t)d * 2, (uint64_t)n_q * d * 2, (uint64_t)batch * heads * n_q * d * 2};
  uint32_t qbox64[4] = {64, 64, 1, 1};
  CUtensorMap map_qd64 = rab::make_tmap_bf16(qdo.data_ptr(), 4, qdims, qstr, qbox64, rab::TmapSwizzle::B128);
  CUtensorMap map_kv = make_kv_map(kv_buf, p, p.hop_owner[0]);
  // dQ accumulator: 2-D (d, b*h*n_pad) fp32, box 32 columns x 32 rows, no swizzle (rows written lane-contiguous)
  uint64_t adims[2] = {(uint64_t)d, (uint64_t)batch * heads * n_pad};
  uint64_t astr[1] = {(uint64_t)d * 4};
  uint32_t abox[2] = {32, 32};
  CUtensorMap map_dq = rab::make_tmap_f32(dq_acc.data_ptr(), 2, adims, astr, abox, rab::TmapSwizzle::None);

  Tensor dk, dv;
  if (dkv_acc_ptrs.empty()) {
    dk = torch::empty({batch, n_k, kv_heads, d}, kv_buf.options());
    dv = torch::empty({batch, n_k, kv_heads, d}, kv_buf.options());
    p.dk = dk.data_ptr();
    p.dv = dv.data_ptr();
    p.ring_reduce = 0;
  } else {
    TORCH_CHECK((int)dkv_acc_ptrs.size() == world && nk_pad % 128 == 0 && nk_pad >= n_k);
    dk = torch::empty({0}, kv_buf.options());
    dv = torch::empty({0}, kv_buf.options());
    p.ring_reduce = 1;
    uint64_t ddims[2] = {(uint64_t)d, (uint64_t)2 * batch * kv_heads * nk_pad};
    uint64_t dstr[1] = {(uint64_t)d * 4};
    uint32_t dbox[2] = {32, 32};
    for (int o = 0; o < world; ++o)
      p.map_dkv[o] = rab::make_tmap_f32(reinterpret_cast<const void*>(dkv_acc_ptrs[o]), 2, ddims, dstr, dbox,
                                        rab::TmapSwizzle::B128);
  }
  rab::launch_attn_bwd_fused(map_qd64, map_kv, map_dq, p, sm_count(), stream);
  return {dk, dv};
}

// acc fp32 [b*h][n_pad][d] -> out 16 bit [b][n][h][d] * scale
void acc_convert(const Tensor& acc, Tensor out, double scale) {
  TORCH_CHECK(acc.is_cuda() && acc.scalar_type() == at::kFloat && acc.is_contiguous() && acc.dim() == 3);
  check_16bit(out, "out");
  TORCH_CHECK(out.is_contiguous() && out.dim() == 4);
  const int b = out.size(0), n = out.size(1), h = out.size(2), d = out.size(3);
  TORCH_CHECK(acc.size(0) == b * h && acc.size(1) >= n && acc.size(2) == d && d % 8 == 0);
  c10::cuda::CUDAGuard guard(acc.device());
  rab::launch_acc_convert(acc.data_ptr<float>(), out.data_ptr(), b, h, n, (int)acc.size(1), d, (float)scale,
                          out.scalar_type() == at::kBFloat16, at::cuda::getCurrentCUDAStream());
}

// ---------------------------------------------------------------------------------------------
// tree-attention decode: ONE persistent cooperative kernel (split-KV partials, in-kernel merge of the splits, publish,
// cross-rank signal, merge over NVLink loads or NVLS multimem reductions).  Every buffer is owned by the caller
// (ops/tree_decode_cuda.py caches them), so the call allocates nothing and can be captured in a CUDA graph.
// ---------------------------------------------------------------------------------------------
int64_t tree_decode_max_ctas(int64_t d, int64_t kv_kind, bool tensor_core) {
  if (tensor_core) return rab::tree_decode_tc_max_ctas((int)kv_kind, sm_count());
  return rab::tree_decode_max_ctas((int)d, (int)kv_kind, sm_count());
}

void tree_decode(const Tensor& q, const c10::optional<Tensor>& k, const c10::optional<Tensor>& v,
                 const c10::optional<Tensor>& k_scale, const c10::optional<Tensor>& v_scale, Tensor scratch,
                 Tensor group_done, Tensor counters, at::IntArrayRef partial_ptrs, int64_t aux_local_ptr,
                 at::IntArrayRef pad_ptrs, int64_t mc_partial_ptr, int64_t mc_aux_ptr, int64_t rank, Tensor out,
                 int64_t kv_heads, int64_t splits, double scale, int64_t scale_block_keys, double eps, int64_t grid,
                 bool tensor_core) {
  TORCH_CHECK(q.is_cuda() && q.is_contiguous() && q.dim() == 3, "q must be contiguous [b, h, d]");
  const int b = q.size(0), h = q.size(1), d = q.size(2);
  TORCH_CHECK(d == 64 || d == 128, "tree decode supports head dim 64 or 128");
  rab::TreeDecodeParams p;
  std::memset(&p, 0, sizeof(p));
  p.q = q.data_ptr();
  p.q_kind = q.scalar_type() == at::kBFloat16 ? 0 : (q.scalar_type() == at::kHalf ? 1 : 2);
  TORCH_CHECK(p.q_kind != 2 || q.scalar_type() == at::kFloat, "q must be bf16, fp16 or fp32");
  int n = 0;
  int64_t kv_plane_stride = 0;  // elements between consecutive (batch, kv head) planes
  if (k.has_value()) {
    TORCH_CHECK(v.has_value() && k->dim() == 4 && k->sizes() == v->sizes());
    TORCH_CHECK(k->is_contiguous() ? v->is_contiguous() : k->strides() == v->strides(), "k and v must share a layout");
    TORCH_CHECK(k->size(0) == b && k->size(1) == kv_heads && k->size(3) == d);
    n = k->size(2);
    // a growing cache passes the filled prefix [b, hk, :n, d] of a [b, hk, capacity, d] buffer: rows stay dense, the
    // (batch, head) planes keep the buffer's stride.  Only the tensor-core kernel takes that (it sees K / V through
    // tensor maps); the CUDA-core kernel needs dense planes.
    const bool rows_dense = k->stride(3) == 1 && k->stride(2) == d && k->stride(0) == kv_heads * k->stride(1) &&
                            k->stride(1) >= (int64_t)n * d;
    TORCH_CHECK(k->is_contiguous() || (tensor_core && rows_dense),
                "k / v must be contiguous [b, hk, n, d] (or, for the tensor-core kernel, a prefix view of a [b, hk, "
                "capacity, d] buffer)");
    kv_plane_stride = k->is_contiguous() ? (int64_t)n * d : k->stride(1);  // strides of size-1 dims are arbitrary
    if (k->scalar_type() == at::kBFloat16) p.kv_kind = 0;
    else if (k->scalar_type() == at::kHalf) p.kv_kind = 1;
    else if (k->scalar_type() == at::kFloat8_e4m3fn) p.kv_kind = 2;
    else TORCH_CHECK(false, "k/v must be bf16, fp16 or float8_e4m3fn");
    TORCH_CHECK(v->scalar_type() == k->scalar_type());
    p.k = k->data_ptr();
    p.v = v->data_ptr();
  }
  p.n_scale_blocks = 1;
  p.scale_block = 1 << 30;  // per-head scales: the whole shard is one block
  if (k_scale.has_value()) {
    TORCH_CHECK(v_scale.has_value() && k_scale->sizes() == v_scale->sizes(), "k_scale and v_scale come together");
    TORCH_CHECK(k_scale->scalar_type() == at::kFloat && v_scale->scalar_type() == at::kFloat);
    TORCH_CHECK(k_scale->is_contiguous() && v_scale->is_contiguous() && k_scale->numel() % (b * kv_heads) == 0);
    p.n_scale_blocks = k_scale->numel() / (b * kv_heads);
    p.k_scale = k_scale->data_ptr<float>();
    p.v_scale = v_scale->data_ptr<float>();
    if (p.n_scale_blocks > 1) {
      TORCH_CHECK(scale_block_keys > 0 && scale_block_keys % 64 == 0, "scale_block_keys must be a multiple of 64");
      TORCH_CHECK((int64_t)p.n_scale_blocks * scale_block_keys >= n, "not enough scale blocks for the shard");
      p.scale_block = (int)scale_block_keys;
    }
  }
  p.batch = b; p.heads = h; p.kv_heads = (int)kv_heads; p.n = n; p.splits = (int)splits;
  TORCH_CHECK(h % kv_heads == 0 && splits >= 1);
  p.scale_log2 = (float)(scale * 1.4426950408889634);
  const int g = h / (int)kv_heads;
  TORCH_CHECK(scratch.scalar_type() == at::kFloat && scratch.is_contiguous() &&
              scratch.numel() >= (int64_t)b * kv_heads * splits * g * (d + 4));
  TORCH_CHECK(group_done.scalar_type() == at::kInt && group_done.numel() >= (int64_t)b * kv_heads * ((g + 3) / 4));
  TORCH_CHECK(counters.scalar_type() == at::kInt && counters.numel() >= 4);
  p.scratch = scratch.data_ptr<float>();
  p.group_done = reinterpret_cast<uint32_t*>(group_done.data_ptr<int>());
  p.counters = reinterpret_cast<uint32_t*>(counters.data_ptr<int>());
  p.world = (int)partial_ptrs.size();
  p.rank = (int)rank;
  TORCH_CHECK(p.world >= 1 && p.world <= rab::kMaxWorld && p.rank < p.world && (int)pad_ptrs.size() == p.world);
  for (int i = 0; i < p.world; ++i) {
    p.partials[i] = reinterpret_cast<const float*>(partial_ptrs[i]);
    p.pads[i] = reinterpret_cast<uint32_t*>(pad_ptrs[i]);
  }
  p.partial_local = const_cast<float*>(p.partials[p.rank]);
  p.aux_local = reinterpret_cast<float*>(aux_local_ptr);
  p.mc_partial = reinterpret_cast<const float*>(mc_partial_ptr);
  p.mc_aux = reinterpret_cast<const float*>(mc_aux_ptr);
  TORCH_CHECK(out.is_cuda() && out.is_contiguous() && out.numel() == (int64_t)b * h * d);
  p.out = out.data_ptr();
  p.out_kind = out.scalar_type() == at::kBFloat16 ? 1 : (out.scalar_type() == at::kHalf ? 0 : 2);
  TORCH_CHECK(p.out_kind != 2 || out.scalar_type() == at::kFloat);
  p.eps = (float)eps;
  c10::cuda::CUDAGuard guard(q.device());
  if (tensor_core) {
    TORCH_CHECK(d == 128 && n > 0, "the tcgen05 decode kernel needs head dim 128 and a non-empty shard");
    // K, V [b*hk, n, d] -> dims (d, n, b*hk); box = one 128-byte wide, 128-key sub-tile
    const uint64_t eb = p.kv_kind == 2 ? 1 : 2;
    uint64_t dims[3] = {(uint64_t)d, (uint64_t)n, (uint64_t)b * kv_heads};
    uint64_t strides[2] = {(uint64_t)d * eb, (uint64_t)kv_plane_stride * eb};
    TORCH_CHECK(strides[1] % 16 == 0, "k / v plane stride must be a multiple of 16 bytes");
    uint32_t box[3] = {(uint32_t)(128 / eb), 128, 1};
    auto mk = [&](const void* base) {
      if (p.kv_kind == 2) return rab::make_tmap_u8(base, 3, dims, strides, box, rab::TmapSwizzle::B128);
      if (p.kv_kind == 1) return rab::make_tmap_f16(base, 3, dims, strides, box, rab::TmapSwizzle::B128);
      return rab::make_tmap_bf16(base, 3, dims, strides, box, rab::TmapSwizzle::B128);
    };
    CUtensorMap map_k = mk(p.k), map_v = mk(p.v);
    rab::launch_tree_decode_tc(map_k, map_v, p, (int)grid, at::cuda::getCurrentCUDAStream());
  } else {
    rab::launch_tree_decode(p, d, (int)grid, at::cuda::getCurrentCUDAStream());
  }
}

void pack_kv(const Tensor& k, const Tensor& v, Tensor slot, int64_t which) {
  check_16bit(k, "k");
  check_16bit(v, "v");
  TORCH_CHECK(k.dim() == 4 && v.dim() == 4 && k.sizes() == v.sizes());
  TORCH_CHECK(k.stride(3) == 1 && v.stride(3) == 1, "k/v need unit stride on the head dim");
  const int b = k.size(0), n = k.size(1), hk = k.size(2), d = k.size(3);
  TORCH_CHECK(d % 8 == 0);
  for (int i = 0; i < 3; ++i)
    TORCH_CHECK(k.stride(i) % 8 == 0 && v.stride(i) % 8 == 0, "k/v strides must be multiples of 8 elements");
  TORCH_CHECK(slot.is_contiguous() && slot.numel() == 2ll * b * n * hk * d && slot.scalar_type() == k.scalar_type());
  c10::cuda::CUDAGuard guard(k.device());
  TORCH_CHECK(which >= 1 && which <= 3, "which: 1 = K half, 2 = V half, 3 = both");
  rab::launch_pack_kv(k.data_ptr(), v.data_ptr(), slot.data_ptr(), b, n, hk, d, k.stride(0), k.stride(1), k.stride(2),
                      v.stride(0), v.stride(1), v.stride(2), (int)which, at::cuda::getCurrentCUDAStream());
}

// x [b, n, h, d] 16 bit (unit stride on d) -> out, rotated by angles [n, >= d/2] fp32 (sign -1: inverse rotation).
//   head_major = false: out [b, n, h, d_out] (d_out >= d: the caller pre-zeroes the padding columns)
//   head_major = true : out [b*h, n, d_out]  (one half of a K/V gather slot)
void rotary(const Tensor& x, const Tensor& angles, Tensor out, bool head_major, double sign) {
  check_16bit(x, "x");
  TORCH_CHECK(x.dim() == 4 && x.stride(3) == 1 && out.is_contiguous() && out.scalar_type() == x.scalar_type());
  const int b = x.size(0), n = x.size(1), h = x.size(2), d = x.size(3);
  TORCH_CHECK(d % 16 == 0, "rotary kernel needs head dim % 16 == 0");
  TORCH_CHECK(angles.is_cuda() && angles.scalar_type() == at::kFloat && angles.dim() == 2 && angles.size(0) == n &&
              angles.size(1) >= d / 2 && angles.stride(1) == 1);
  for (int i = 0; i < 3; ++i) TORCH_CHECK(x.stride(i) % 8 == 0, "x strides must be multiples of 8 elements");
  const int d_out = out.size(-1);
  TORCH_CHECK(d_out >= d && d_out % 8 == 0 && out.numel() == (int64_t)b * n * h * d_out);
  long long ob, on, oh;
  if (head_major) { ob = (long long)h * n * d_out; oh = (long long)n * d_out; on = d_out; }
  else { ob = (long long)n * h * d_out; on = (long long)h * d_out; oh = d_out; }
  c10::cuda::CUDAGuard guard(x.device());
  rab::launch_rotary(x.data_ptr(), out.data_ptr(), angles.data_ptr<float>(), (int)angles.stride(0), b, n, h, d,
                     x.stride(0), x.stride(1), x.stride(2), ob, on, oh, (float)sign,
                     x.scalar_type() == at::kBFloat16, at::cuda::getCurrentCUDAStream());
}

void device_barrier(at::IntArrayRef pad_ptrs, int64_t rank, int64_t epoch) {
  rab::BarrierParams p;
  std::memset(&p, 0, sizeof(p));
  p.world = (int)pad_ptrs.size();
  TORCH_CHECK(p.world <= rab::kMaxWorld);
  p.rank = (int)rank;
  p.epoch = (uint32_t)epoch;
  for (int i = 0; i < p.world; ++i) p.pads[i] = reinterpret_cast<uint32_t*>(pad_ptrs[i]);
  rab::launch_device_barrier(p, at::cuda::getCurrentCUDAStream());
}

// ---------------------------------------------------------------------------------------------
// symmetric memory
// ---------------------------------------------------------------------------------------------
std::tuple<Tensor, Tensor> symm_alloc(int64_t bytes) {
  Tensor handle = torch::empty({rab::kIpcHandleBytes}, torch::dtype(torch::kUInt8));
  void* base = rab::symm_alloc((size_t)bytes, handle.data_ptr<uint8_t>());
  int dev = 0;
  cudaGetDevice(&dev);
  Tensor t = torch::from_blob(
      base, {bytes}, [base](void*) { rab::symm_free(base); },
      torch::TensorOptions().dtype(torch::kUInt8).device(torch::kCUDA, dev));
  return {t, handle};
}

void peer_copy(Tensor dst, int64_t src_ptr, int64_t nbytes) {
  TORCH_CHECK(dst.is_cuda() && dst.is_contiguous() && (int64_t)dst.nbytes() >= nbytes);
  c10::cuda::CUDAGuard guard(dst.device());
  rab::cuda_check(cudaMemcpyAsync(dst.data_ptr(), reinterpret_cast<const void*>(src_ptr), (size_t)nbytes,
                                  cudaMemcpyDeviceToDevice, at::cuda::getCurrentCUDAStream()),
                  "peer_copy");
}

// Stream-ordered 32-bit flag write (cuStreamWriteValue32): a memory operation of the stream itself, no kernel and no
// copy-engine job.  The backward uses it to publish "K/V slot o has landed" from the side stream while its persistent
// kernel owns every SM (a flag written by a kernel could never be scheduled next to it).
void stream_write_u32(Tensor flags, int64_t index, int64_t value) {
  TORCH_CHECK(flags.is_cuda() && flags.scalar_type() == at::kInt && flags.is_contiguous() && index >= 0 &&
              index < flags.numel());
  c10::cuda::CUDAGuard guard(flags.device());
  rab::stream_write_value32(flags.data_ptr<int>() + index, (uint32_t)value, at::cuda::getCurrentCUDAStream());
}

int64_t symm_open(const Tensor& handle) {
  TORCH_CHECK(!handle.is_cuda() && handle.scalar_type() == torch::kUInt8 && handle.numel() == rab::kIpcHandleBytes);
  return reinterpret_cast<int64_t>(rab::symm_open(handle.contiguous().data_ptr<uint8_t>()));
}

void symm_close(int64_t ptr) { rab::symm_close(reinterpret_cast<void*>(ptr)); }

}  // namespace

TORCH_LIBRARY(rab, m) {
  m.def("umma_rate(int mode, int n, int reps, int alt, int ctas) -> Tensor");
  m.def("umma_probe(Tensor a, Tensor b, int mode, int n, int k, int idesc, int a_lbo, int a_sbo, int b_lbo, int "
        "b_sbo, int b_kstep) -> Tensor");
  m.def("attn_fwd(Tensor q, Tensor kv_buf, int[] peer_ptrs, Tensor ready, " PROBLEM_SCHEMA ") -> (Tensor, Tensor)");
  m.def("attn_fwd_hop(Tensor q, Tensor kv_slot, Tensor(a!) carry_o, Tensor(b!) carry_ml, bool carry_in, bool carry_out, "
        PROBLEM_SCHEMA ") -> (Tensor, Tensor)");
  m.def("pack_kv(Tensor k, Tensor v, Tensor(a!) slot, int which=3) -> ()");
  m.def("rotary(Tensor x, Tensor angles, Tensor(a!) out, bool head_major, float sign) -> ()");
  m.def("tree_decode(Tensor q, Tensor? k, Tensor? v, Tensor? k_scale, Tensor? v_scale, Tensor(a!) scratch, Tensor(b!) "
        "group_done, Tensor(c!) counters, int[] partial_ptrs, int aux_local_ptr, int[] pad_ptrs, int mc_partial_ptr, int "
        "mc_aux_ptr, int rank, Tensor(d!) out, int kv_heads, int splits, float scale, int scale_block_keys, float eps, "
        "int grid, bool tensor_core) -> ()");
  m.def("tree_decode_max_ctas(int d, int kv_kind, bool tensor_core) -> int");
  m.def("bwd_prep(Tensor q, Tensor o, Tensor dout, Tensor lse, Tensor(a!) qdo_buf, Tensor(b!) stat_buf, int rank) -> ()");
  m.def("attn_bwd_dq(Tensor qdo_buf, Tensor kv_buf, Tensor stat_buf, Tensor? ready, int ready_target, " PROBLEM_SCHEMA
        ") -> Tensor");
  m.def("attn_bwd_dkdv(Tensor qdo_buf, Tensor kv_buf, Tensor stat_buf, Tensor? ready, int ready_target, " PROBLEM_SCHEMA
        ") -> (Tensor, Tensor)");
  m.def("attn_bwd_dq_hop(Tensor qdo_own, Tensor kv_slot, Tensor stat_own, Tensor(a!) carry, bool carry_in, bool "
        "carry_out, " PROBLEM_SCHEMA ") -> Tensor");
  m.def("attn_bwd_dkdv_hop(Tensor qdo_slot, Tensor kv_own, Tensor stat_slot, Tensor(a!) carry, bool carry_in, bool "
        "carry_out, " PROBLEM_SCHEMA ") -> (Tensor, Tensor)");
  m.def("attn_bwd_ring(Tensor qdo, Tensor kv_buf, Tensor stat, Tensor(a!) dq_acc, Tensor? ready, int ready_target, int[] "
        "dkv_acc_ptrs, int nk_pad, " PROBLEM_SCHEMA ") -> (Tensor, Tensor)");
  m.def("acc_convert(Tensor acc, Tensor(a!) out, float scale) -> ()");
  m.def("set_fetch_timing(Tensor? times) -> ()");
  m.def("device_barrier(int[] pad_ptrs, int rank, int epoch) -> ()");
  m.def("peer_copy(Tensor(a!) dst, int src_ptr, int nbytes) -> ()");
  m.def("stream_write_u32(Tensor(a!) flags, int index, int value) -> ()");
  m.def("symm_alloc(int bytes) -> (Tensor, Tensor)");
  m.def("symm_open(Tensor handle) -> int");
  m.def("symm_close(int ptr) -> ()");
}

TORCH_LIBRARY_IMPL(rab, CUDA, m) {
  m.impl("umma_probe", &umma_probe);
  m.impl("attn_fwd", &attn_fwd);
  m.impl("attn_fwd_hop", &attn_fwd_hop);
  m.impl("pack_kv", &pack_kv);
  m.impl("rotary", &rotary);
  m.impl("tree_decode", &tree_decode);
  m.impl("bwd_prep", &bwd_prep);
  m.impl("attn_bwd_dq", &attn_bwd_dq);
  m.impl("attn_bwd_dkdv", &attn_bwd_dkdv);
  m.impl("attn_bwd_dq_hop", &attn_bwd_dq_hop);
  m.impl("attn_bwd_dkdv_hop", &attn_bwd_dkdv_hop);
  m.impl("attn_bwd_ring", &attn_bwd_ring);
  m.impl("acc_convert", &acc_convert);
}

TORCH_LIBRARY_IMPL(rab, CompositeExplicitAutograd, m) {
  m.impl("umma_rate", &umma_rate);
  m.impl("set_fetch_timing", &set_fetch_timing);
  m.impl("device_barrier", &device_barrier);
  m.impl("peer_copy", &peer_copy);
  m.impl("stream_write_u32", &stream_write_u32);
  m.impl("tree_decode_max_ctas", &tree_decode_max_ctas);
  m.impl("symm_alloc", &symm_alloc);
  m.impl("symm_open", &symm_open);
  m.impl("symm_close", &symm_close);
}
