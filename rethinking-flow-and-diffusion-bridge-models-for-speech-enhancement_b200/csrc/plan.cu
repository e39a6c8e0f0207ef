// The NCSN++ forward as a static launch plan (fdbm/backbones/ncsnpp_v2.py:241-401 and
// ncsnpp_v2_predictive.py:222-362), plus the N-step sampler loop of fdbm/bridge.py:66-113.
//
// fdbm_plan_create walks the reference constructor's module list (ncsnpp_v2.py:95-239) once for a
// fixed (batch, n_frames) and records, in execution order, every kernel launch with its buffers
// resolved inside one device arena (first-fit with explicit frees, so the skip stack and the
// temporaries of a residual block reuse memory).  Forward / sampler replay that list; the sampler
// captures all N steps (backbone + bridge update) into one CUDA graph per argument set.
#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>
#include "common.cuh"

using namespace fdbm;

namespace {

struct Mod {
  enum Kind { FOURIER, LINEAR, CONV3, RES, ATTN, COMBINE, GN } kind;
  int idx, cin, cout;
  bool up, down;
};

struct Slot { int64_t off; int64_t numel; bool loaded; };     // fp32 parameter inside `params`

struct Act {                 // one residual-stream tensor [B,T,F,C]: 16-bit GEMM-operand copy, channel sums
  op_t* h16 = nullptr;
  double* sums = nullptr;
  float* grad = nullptr;      // training plans: fp32 gradient accumulator (loss-scaled), zeroed at the start of backward
  int C = 0, T = 0, F = 0;
};

struct GraphKey {
  const void* p[6]; int n_steps, kind; uint64_t seed;
  bool operator==(const GraphKey& o) const {
    for (int i = 0; i < 6; ++i) if (p[i] != o.p[i]) return false;
    return n_steps == o.n_steps && kind == o.kind && seed == o.seed;
  }
};

// first-fit arena over one cudaMalloc
class Arena {
 public:
  void reset(int64_t cap) { free_.clear(); free_[0] = cap; cap_ = cap; peak_ = 0; }
  int64_t alloc(int64_t bytes) {
    bytes = (bytes + 1023) / 1024 * 1024;
    for (auto it = free_.begin(); it != free_.end(); ++it) {
      if (it->second >= bytes) {
        const int64_t off = it->first, rest = it->second - bytes;
        free_.erase(it);
        if (rest) free_[off + bytes] = rest;
        live_[off] = bytes;
        peak_ = std::max(peak_, off + bytes);
        return off;
      }
    }
    return -1;
  }
  void release(int64_t off) {
    auto it = live_.find(off);
    if (it == live_.end()) return;
    int64_t o = off, n = it->second;
    live_.erase(it);
    auto nx = free_.lower_bound(o);
    if (nx != free_.end() && o + n == nx->first) { n += nx->second; nx = free_.erase(nx); }
    if (nx != free_.begin()) {
      auto pv = std::prev(nx);
      if (pv->first + pv->second == o) { o = pv->first; n += pv->second; free_.erase(pv); }
    }
    free_[o] = n;
  }
  int64_t peak() const { return peak_; }
 private:
  std::map<int64_t, int64_t> free_, live_;
  int64_t cap_ = 0, peak_ = 0;
};

__global__ void add_vec_kernel(const float* a, const float* b, float* o, int n) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) o[i] = a[i] + (b ? b[i] : 0.f);
}

}  // namespace

struct fdbm_plan {
  fdbm_arch arch;
  int B = 0, T = 0, F = 0, F_io = 257, Cin = 4;
  std::vector<Mod> mods;
  // parameters
  std::unordered_map<std::string, Slot> slots;
  int64_t params_numel = 0;
  float* params = nullptr;            // fp32 originals + derived fp32 (combined biases)
  op_t* wpacked = nullptr;   // packed conv weights
  int64_t wpacked_bytes = 0;
  int dense_rows = 0;
  bool weights_ready = false;
  // activations
  uint8_t* arena = nullptr;
  int64_t arena_bytes = 0;
  int64_t sums_pool_bytes = 0;
  // per-call arguments the recorded ops read
  const float* cur_x = nullptr; const float* cur_y = nullptr; const float* cur_t = nullptr; int cur_t_stride = 1;
  float* cur_out = nullptr;
  float* d_buf = nullptr;             // backbone output inside the sampler loop
  std::vector<std::function<int(cudaStream_t)>> ops;        // one forward: exactly one kernel launch per entry
  std::vector<int> op_kind;                                  // FDBM_OP_* of every entry
  std::vector<double> op_flops;                              // algorithmic FLOPs (2*MAC) of every entry (convs)
  std::vector<std::function<int(cudaStream_t)>> pack_ops;   // weight packing after load_weights (the few odd ones)
  // training: per-site gradient sums (common.cuh DeferDesc): one pool, one memset per backward, one reduction launch
  double* defer_pool = nullptr; int64_t defer_pool_bytes = 0;
  std::vector<DeferDesc> defer_descs; DeferDesc* defer_descs_d = nullptr;
  std::vector<PackDesc> pack_descs;                          // ... and all regular conv packs, run as ONE launch
  PackDesc* pack_descs_d = nullptr; long long pack_blocks = 0;
  int n_launches = 0;
  // training (fdbm_plan_create_train): nothing in the arena is reused, every forward tensor stays live for backward
  bool train = false;
  float* grads = nullptr;              // flat fp32 parameter gradients, same layout as `params`
  op_t* wpacked_d = nullptr;           // dgrad packs (weights transposed + flipped)
  int64_t wpacked_d_bytes = 0;
  float* wgrad_ws = nullptr;           // split partials of the wgrad kernel
  int64_t wgrad_ws_bytes = 0;
  std::vector<std::function<int(cudaStream_t)>> bwd_ops;
  std::vector<int> bwd_kind;
  // Activation-gradient accumulators (fp32, one per residual-stream tensor).  They are not cleared up front: the FIRST
  // contribution of a backward pass writes instead of adding (saves the memset and one read of every tensor per step); an
  // op that can only add, or an op that reads a buffer nobody wrote, clears it on demand.
  std::vector<std::pair<void*, size_t>> zero_list;
  std::unordered_map<const void*, int> gz_index;
  std::vector<uint8_t> gz_written;
  void grads_begin() { gz_written.assign(zero_list.size(), 0); }
  bool grad_first(const float* g) {                     // true exactly once per backward pass and buffer
    auto it = gz_index.find(g);
    if (it == gz_index.end() || gz_written[it->second]) return false;
    gz_written[it->second] = 1;
    return true;
  }
  int grad_ensure(const float* g, cudaStream_t s) {     // before an add-only writer or a reader
    if (!grad_first(g)) return FDBM_OK;
    const auto& z = zero_list[gz_index[g]];
    FDBM_CUDA(cudaMemsetAsync(z.first, 0, z.second, s));
    return FDBM_OK;
  }
  const float* cur_gout = nullptr;     // dL/dD of the current backward call (loss-scaled), cplx [B,1,257,T]
  float cur_inv = 1.0f;                // 1 / loss scale
  float* adam_m = nullptr; float* adam_v = nullptr; float* ema = nullptr; double* opt_scratch = nullptr;
  double* opt_state = nullptr;         // {applied updates, skipped steps, last gradient norm, reserved}
  float* ema_backup = nullptr;         // live parameters parked here while the EMA is swapped in
  bool ema_swapped = false;
  int n_bwd_launches = 0;
  int device = 0;                      // the device the plan's memory lives on; every entry point checks it is current
  // sampler staging (bridge inference plans, allocated by fdbm_plan_create): the captured graph reads these fixed buffers
  static constexpr int kMaxSteps = 1024;
  static constexpr int kRing = 8;
  float* smp_y = nullptr; float* smp_x = nullptr; float* smp_times = nullptr; float* smp_coef = nullptr; uint64_t* smp_rng = nullptr;
  uint8_t* smp_pinned = nullptr;       // kRing host slots of {seed[2], times[kMaxSteps], coef[3 kMaxSteps]}
  cudaEvent_t smp_ev[kRing] = {};
  int smp_pos = 0;
  std::vector<float> smp_h_times, smp_h_coef;
  // graph cache
  bool have_graph = false; GraphKey graph_key{}; cudaGraphExec_t graph_exec = nullptr;
  cudaStream_t capture_stream = nullptr;   // private stream: capture works even when the caller is on the legacy stream
  int64_t extra_bytes = 0;             // device memory outside the arena / params / packs (staging, optimiser, gradients)
};

namespace {
constexpr size_t kSlotBytes = 16 + sizeof(float) * 4 * fdbm_plan::kMaxSteps;

// every plan entry point: the plan's device must be the calling thread's current device (allocations, launches and the
// caller's stream all refer to the current device; a mismatch would fault on foreign pointers)
int plan_guard(const fdbm_plan* plan, const char* who) {
  if (!plan) { set_error("%s: null plan", who); return FDBM_EINVAL; }
  const int dev = current_device();
  if (dev != plan->device) {
    set_error("%s: the plan lives on device %d but the current device is %d (select the tensors' device first)", who, plan->device, dev);
    return FDBM_ESTATE;
  }
  return FDBM_OK;
}
}  // namespace

namespace {

std::vector<Mod> build_modules(const fdbm_arch& a) {
  std::vector<Mod> m;
  auto add = [&](Mod::Kind k, int cin, int cout, bool up = false, bool down = false) {
    m.push_back(Mod{k, static_cast<int>(m.size()), cin, cout, up, down});
  };
  const int nf = a.nf, C = a.predictive ? 2 : 4, L = a.n_levels;
  if (!a.predictive) { add(Mod::FOURIER, 0, nf); add(Mod::LINEAR, 2 * nf, 4 * nf); add(Mod::LINEAR, 4 * nf, 4 * nf); }
  add(Mod::CONV3, C, nf);
  std::vector<int> hs_c{nf};
  int in_ch = nf;
  for (int lvl = 0; lvl < L; ++lvl) {
    const int res = a.image_size >> lvl;
    for (int b = 0; b < a.num_res_blocks; ++b) {
      const int out_ch = nf * a.ch_mult[lvl];
      add(Mod::RES, in_ch, out_ch);
      in_ch = out_ch;
      if (res == a.attn_resolution) add(Mod::ATTN, in_ch, in_ch);
      hs_c.push_back(in_ch);
    }
    if (lvl != L - 1) {
      add(Mod::RES, in_ch, in_ch, false, true);
      add(Mod::COMBINE, C, in_ch);
      hs_c.push_back(in_ch);
    }
  }
  in_ch = hs_c.back();
  add(Mod::RES, in_ch, in_ch); add(Mod::ATTN, in_ch, in_ch); add(Mod::RES, in_ch, in_ch);
  for (int lvl = L - 1; lvl >= 0; --lvl) {
    const int res = a.image_size >> lvl;
    for (int b = 0; b < a.num_res_blocks + 1; ++b) {
      const int out_ch = nf * a.ch_mult[lvl];
      add(Mod::RES, in_ch + hs_c.back(), out_ch);
      hs_c.pop_back();
      in_ch = out_ch;
    }
    if (res == a.attn_resolution) add(Mod::ATTN, in_ch, in_ch);
    add(Mod::GN, in_ch, in_ch);
    add(Mod::CONV3, in_ch, C);
    if (lvl != 0) add(Mod::RES, in_ch, in_ch, true, false);
  }
  return m;
}

struct Builder {
  fdbm_plan* P;
  Arena arena;
  int64_t wp_off = 0;                  // running offset (bytes) into wpacked
  int dense_off = 0;                   // running row offset into the Dense_0 table
  bool dry = true;                     // first pass: sizes only
  // every GroupNorm-statistics buffer is a slice of one pool that a single memset zeroes at the start of the forward (the
  // per-convolution memsets were ~100 extra stream operations on the critical path; training plans keep the slices for the backward)
  uint8_t* sums_pool = nullptr;
  int64_t sums_used = 0;

  // ---------------- training: backward ops are recorded per forward composite ("group") and replayed in reverse
  typedef std::function<int(cudaStream_t)> Op;
  std::vector<std::vector<std::pair<Op, int>>> groups;
  int64_t wd_off = 0;                  // running offset (bytes) into wpacked_d
  int64_t ws_need = 0;                 // largest wgrad workspace
  op_t *T1 = nullptr, *T2 = nullptr, *T3 = nullptr, *T4 = nullptr, *T5 = nullptr;     // shared backward scratch (16-bit)
  double *Sbuf = nullptr, *sumsA = nullptr;
  float *att_scratch = nullptr, *d_dense = nullptr, *g_temb = nullptr;
  const float* zero_bias = nullptr;
  bool train() const { return P->train; }
  int64_t defer_used = 0;
  double* site_sums(int64_t n_doubles) {                 // this site's slice of the deferred-sums pool (zero at the start of a backward)
    const int64_t bytes = (n_doubles * 8 + 255) / 256 * 256;
    defer_used += bytes;
    if (dry) return reinterpret_cast<double*>(P->arena);  // sizing pass: only counted
    return reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(P->defer_pool) + defer_used - bytes);
  }
  void defer_col_sums(const double* src, int C, int64_t dst_off, float* per_b = nullptr, int per_b_ld = 0) {
    if (!dry) P->defer_descs.push_back(DeferDesc{src, P->B, C, 0, dst_off >= 0 ? P->grads + dst_off : nullptr, nullptr, per_b, per_b_ld});
  }
  void defer_gn_param(const double* S, int C, int64_t gamma_off, int64_t beta_off) {
    if (!dry) P->defer_descs.push_back(DeferDesc{S, P->B, C, 1, P->grads + gamma_off, P->grads + beta_off, nullptr, 0});
  }
  void bgroup() { if (train()) groups.emplace_back(); }
  void bop(Op f, int kind = FDBM_OP_NORM) { if (train() && !dry) groups.back().emplace_back(std::move(f), kind); }
  float* gp(int64_t off) const { return P->grads + off; }
  float* galloc(int64_t n) {
    float* g = alloc<float>(n);
    if (!dry) { P->gz_index[g] = static_cast<int>(P->zero_list.size()); P->zero_list.emplace_back(g, static_cast<size_t>(n) * sizeof(float)); }
    return g;
  }
  op_t* pack_d(int64_t w_off, int Cout, int Cin, int ksize, int Cin_total = 0, int ci_off = 0, op_t* into = nullptr) {
    const int k = ksize == -1 ? 1 : ksize;
    op_t* dst = into;
    if (!dst) {
      dst = reinterpret_cast<op_t*>(reinterpret_cast<uint8_t*>(P->wpacked_d) + wd_off);
      wd_off += (conv_wpack_bytes(Cout, k, 0, Cin) + 1023) / 1024 * 1024;
    }
    const float* w = pp(w_off);
    if (!dry) P->pack_descs.push_back(pack_desc_dgrad(w, Cout, Cin, ksize, dst, Cin_total, ci_off));
    return dst;
  }
  // dX (+)= conv(dY, W'): 16-bit output and/or fp32 in-place accumulation
  void dgrad_op(const op_t* dy, int Cdy, int taps, const op_t* wd, int Cdx, int T, int F, op_t* out16, float* acc) {
    ConvArgs c;
    c.seg[0] = seg(dy, Cdy, taps); c.n_seg = 1;
    c.wpack = wd; c.bias = zero_bias; c.residual = acc; c.scale = 1.0f;
    c.B = P->B; c.T = T; c.F = F; c.Cout = Cdx; c.out_f32 = acc; c.out_h16 = out16;
    fdbm_plan* plp = P;
    bop([=](cudaStream_t s) {
      ConvArgs cc = c;
      if (acc && plp->grad_first(acc)) cc.residual = nullptr;     // first contribution: write, do not read-add
      return launch_conv_igemm(cc, s);
    }, FDBM_OP_CONV);
  }
  void wgrad_op(WgradCall c, int64_t dw_off) {
    c.B = P->B;
    ws_need = std::max(ws_need, conv_wgrad_workspace_bytes(c.Cout, c.Cin, c.ksize, c.B, c.T, c.F));
    fdbm_plan* plp = P;
    bop([=](cudaStream_t s) {
      WgradCall cc = c;
      cc.scale = plp->cur_inv; cc.dw = plp->grads + dw_off; cc.workspace = plp->wgrad_ws;
      return launch_conv_wgrad_ex(cc, s);
    }, FDBM_OP_WGRAD);
  }
  // GroupNorm(+SiLU) backward of one normalised (possibly concatenated) tensor: g_a [B,P,Ctot] 16-bit -> x.grad +=
  void gn_bwd(const op_t* g_a, const Act& x1, const Act* x2, const float2* tab, const float2* stats, int64_t gw_off,
              int64_t gb_off, int act) {
    const int B = P->B, C1 = x1.C, C2 = x2 ? x2->C : 0, Ct = C1 + C2;
    const int64_t px = static_cast<int64_t>(x1.T) * x1.F;
    const float* gamma = pp(gw_off);
    double* S = site_sums(static_cast<int64_t>(B) * Ct * 2);
    defer_gn_param(S, Ct, gw_off, gb_off);
    fdbm_plan* plp = P;
    const Act a1 = x1; const Act a2 = x2 ? *x2 : Act();
    // one reduce + apply launch pair over the whole batch.  Measured: per-utterance chunks small enough for the apply pass to
    // re-read x and g_a from L2 (level 0) made the level-0 GroupNorm backward 2x SLOWER (1.90 vs 0.93 ms: 64 short launches
    // with their tails instead of 4).
    bop([=](cudaStream_t s) {
      const bool f1 = plp->grad_first(a1.grad), f2 = C2 ? plp->grad_first(a2.grad) : false;
      if (int rc = launch_gn_bwd_reduce(g_a, Ct, 0, a1.h16, 1, C1, Ct, 0, tab, stats, act, B, px, S, s)) return rc;
      if (C2) if (int rc = launch_gn_bwd_reduce(g_a, Ct, C1, a2.h16, 1, C2, Ct, C1, tab, stats, act, B, px, S, s)) return rc;
      if (int rc = launch_gn_bwd_apply(g_a, Ct, 0, a1.h16, 1, C1, Ct, 0, tab, stats, gamma, act, B, px, S, a1.grad, nullptr, nullptr, s, f1)) return rc;
      if (C2) if (int rc = launch_gn_bwd_apply(g_a, Ct, C1, a2.h16, 1, C2, Ct, C1, tab, stats, gamma, act, B, px, S, a2.grad, nullptr, nullptr, s, f2)) return rc;
      return FDBM_OK;
    });
  }
  float2* norm_stats(const double* q1) {
    if (!train()) return nullptr;
    if (q1 != last_stats_q1) return nullptr;            // always called right behind norm_table() of the same GroupNorm (build() checks)
    return last_stats;
  }

  // ---------------- parameters
  int64_t param(const std::string& name, int64_t numel) {
    auto it = P->slots.find(name);
    if (it != P->slots.end()) return it->second.off;
    const int64_t off = P->params_numel;
    P->slots[name] = Slot{off, numel, false};
    P->params_numel += (numel + 3) / 4 * 4;              // keep every tensor 16-byte aligned
    return off;
  }
  int64_t derived(int64_t numel) {                       // fp32 scratch parameter (not loaded by name)
    const int64_t off = P->params_numel;
    P->params_numel += (numel + 3) / 4 * 4;
    return off;
  }
  float* pp(int64_t off) const { return P->params + off; }     // call OUTSIDE recorded lambdas only
  std::string pre(const Mod& m) const { return "all_modules." + std::to_string(m.idx) + "."; }

  // ---------------- activations
  template <typename Tp> Tp* alloc(int64_t n_elems) {
    const int64_t off = arena.alloc(n_elems * static_cast<int64_t>(sizeof(Tp)));
    if (off < 0) return nullptr;
    return reinterpret_cast<Tp*>(P->arena + off);
  }
  void release(const void* p) { if (p && !P->train) arena.release(reinterpret_cast<const uint8_t*>(p) - P->arena); }
  double* alloc_sums(int64_t n_doubles) {
    const int64_t bytes = (n_doubles * 8 + 255) / 256 * 256;
    sums_used += bytes;
    if (dry) return reinterpret_cast<double*>(P->arena);          // sizing pass: only counted (the pool is added to the peak)
    return reinterpret_cast<double*>(sums_pool + sums_used - bytes);
  }
  Act new_act(int C, int T, int F) {
    Act a; a.C = C; a.T = T; a.F = F;
    // the residual stream lives in the 16-bit operand format only: the identity shortcut re-reads the 16-bit copy (one
    // rounding per block, which the 1/sqrt(2) of every block keeps from accumulating), and the backward pass of a training
    // plan normalises / recomputes from the same 16-bit tensors the forward convolutions consumed
    a.h16 = alloc<op_t>(static_cast<int64_t>(P->B) * T * F * C);
    a.sums = alloc_sums(static_cast<int64_t>(P->B) * C * 2);
    if (P->train) a.grad = galloc(static_cast<int64_t>(P->B) * T * F * C);
    return a;
  }
  void free_act(Act& a) { release(a.h16); if (train()) release(a.sums); a.h16 = nullptr; a.sums = nullptr; }
  // (scale, shift) table of a GroupNorm over the channel concatenation x1 (+ x2): a tiny launch; the consuming
  // convolution applies it while the operand tile sits in shared memory
  float2* norm_table(const double* q1, int C1, const double* q2, int C2, const float* gamma, const float* beta, int T, int F) {
    const int B = P->B;
    float2* tab = alloc<float2>(static_cast<int64_t>(B) * (C1 + C2));
    const int64_t px = static_cast<int64_t>(T) * F;
    const int blk_real = P->arch.channel_block_real;
    // training plans: the same launch leaves the per-group (mean, rstd) the backward needs (norm_stats() hands them out)
    float2* st = train() ? alloc<float2>(static_cast<int64_t>(B) * 32) : nullptr;
    last_stats = st; last_stats_q1 = q1;
    op([=](cudaStream_t s) { return launch_gn_finalize(q1, C1, q2, C2, gamma, beta, B, px, tab, s, blk_real, st); }, FDBM_OP_STATS);
    return tab;
  }
  float2* last_stats = nullptr; const double* last_stats_q1 = nullptr;
  static ConvSeg seg(const op_t* in, int C, int taps, const float2* tab = nullptr, int tab_stride = 0, int act = 0) {
    ConvSeg sg; sg.in = in; sg.C = C; sg.taps = taps; sg.norm_tab = tab; sg.tab_stride = tab_stride; sg.act = act;
    return sg;
  }

  void op(std::function<int(cudaStream_t)> f, int kind, double flops = 0.0) {
    if (dry) return;
    P->ops.push_back(std::move(f));
    P->op_kind.push_back(kind);
    P->op_flops.push_back(flops);
    P->n_launches += 1;
  }
  // convolution; the channel statistics of its output come out of the same kernel's epilogue
  void conv_op(ConvArgs c, double flops = 0.0) {
    if (flops == 0.0) {
      double k = 0.0;
      for (int i = 0; i < c.n_seg; ++i) k += static_cast<double>(c.seg[i].taps) * c.seg[i].C;
      flops = 2.0 * c.B * c.T * c.F * c.Cout * k;
    }
    c.sums_prezeroed = true;                          // every statistics buffer is a slice of the pool zeroed at the start of the forward
    if (c.bias_b && !train()) {
      fdbm_plan* plp = P;
      op([=](cudaStream_t s) {
        ConvArgs cc = c;
        if (plp->cur_t_stride == 0) cc.bias_b_stride = 0;          // uniform time: all utterances share FiLM row 0
        return launch_conv_igemm(cc, s);
      }, FDBM_OP_CONV, flops);
      return;
    }
    op([=](cudaStream_t s) { return launch_conv_igemm(c, s); }, FDBM_OP_CONV, flops);
  }
  void pack_op(std::function<int(cudaStream_t)> f) { if (!dry) P->pack_ops.push_back(std::move(f)); }

  // packed weights for conv (w1: name, C1, ksize (3, 1 or -1 = NIN [in][out])), optional fused 1x1 w2
  op_t* pack(const std::string& w1, int C1, int ksize, const std::string& w2, int C2, int Cout,
                      int rows_total = 0, int row_off = 0, op_t* into = nullptr) {
    const int k = ksize == -1 ? 1 : ksize;
    if (rows_total == 0) rows_total = Cout;
    op_t* dst = into;
    if (!dst) {
      dst = reinterpret_cast<op_t*>(reinterpret_cast<uint8_t*>(P->wpacked) + wp_off);
      wp_off += (conv_wpack_bytes(C1, k, C2, rows_total) + 1023) / 1024 * 1024;
    }
    const float* p1 = pp(param(w1, static_cast<int64_t>(Cout) * C1 * k * k));
    const float* p2 = C2 ? pp(param(w2, static_cast<int64_t>(Cout) * C2)) : nullptr;
    if (!dry) P->pack_descs.push_back(pack_desc_fwd(p1, C1, ksize, p2, C2, Cout, rows_total, row_off, dst));
    return dst;
  }

  // ---------------- layers
  struct CombineArgs { const float* pyr; const float* w; const float* b; int Cp; int64_t w_off, b_off; };
  // ResnetBlockBigGANpp (layerspp.py:242-274) on the concatenation of x1 (and x2)
  Act resblock(const Mod& m, const Act& x1, const Act* x2, const float* dense, int dense_stride,
               const CombineArgs* comb = nullptr) {
    const int B = P->B, Cin = m.cin, Cout = m.cout;
    const int mode = m.down ? 1 : (m.up ? 2 : 0);
    const int T = x1.T, F = x1.F;
    const int To = mode == 1 ? T / 2 : (mode == 2 ? T * 2 : T), Fo = mode == 1 ? F / 2 : (mode == 2 ? F * 2 : F);
    const bool shortcut = (Cin != Cout) || m.up || m.down;
    const std::string p = pre(m);
    const int64_t o_g0w = param(p + "GroupNorm_0.weight", Cin), o_g0b = param(p + "GroupNorm_0.bias", Cin);
    const int64_t o_c0w = param(p + "Conv_0.weight", static_cast<int64_t>(Cout) * Cin * 9), o_c0b = param(p + "Conv_0.bias", Cout);
    const int64_t o_g1w = param(p + "GroupNorm_1.weight", Cout), o_g1b = param(p + "GroupNorm_1.bias", Cout);
    const int64_t o_c1w = param(p + "Conv_1.weight", static_cast<int64_t>(Cout) * Cout * 9), o_c1b = param(p + "Conv_1.bias", Cout);
    const float* g0w = pp(o_g0w); const float* g0b = pp(o_g0b); const float* c0b = pp(o_c0b);
    const float* g1w = pp(o_g1w); const float* g1b = pp(o_g1b); const float* c1b = pp(o_c1b);
    op_t* w0 = pack(p + "Conv_0.weight", Cin, 3, "", 0, Cout);
    op_t* w1 = shortcut ? pack(p + "Conv_1.weight", Cout, 3, p + "Conv_2.weight", Cin, Cout)
                                 : pack(p + "Conv_1.weight", Cout, 3, "", 0, Cout);
    const float* bias1 = c1b;
    int64_t o_c2w = -1, o_c2b = -1;
    if (shortcut) {                                   // Conv_1.bias + Conv_2.bias, summed once at load time
      o_c2w = param(p + "Conv_2.weight", static_cast<int64_t>(Cout) * Cin);
      o_c2b = param(p + "Conv_2.bias", Cout);
      const float* c2b = pp(o_c2b);
      float* bsum = pp(derived(Cout));
      bias1 = bsum;
      pack_op([=](cudaStream_t s) {
        add_vec_kernel<<<ceil_div(Cout, 256), 256, 0, s>>>(c1b, c2b, bsum, Cout);
        FDBM_LAUNCH_CHECK();
        return FDBM_OK;
      });
    }
    int dense_row = -1;
    if (!P->arch.predictive) {
      param(p + "Dense_0.weight", static_cast<int64_t>(Cout) * 4 * P->arch.nf);   // slots are laid out by build_dense()
      dense_row = dense_off;
      dense_off += Cout;
    }

    const int64_t npx = static_cast<int64_t>(B) * To * Fo;
    const int C1 = x1.C, C2 = x2 ? x2->C : 0;
    // Conv_0 output only feeds GroupNorm_1: keep it in the 16-bit operand format (its statistics are taken
    // from the fp32 accumulators in the conv epilogue, before rounding)
    op_t* h1 = alloc<op_t>(npx * Cout);
    double* h1_sums = alloc_sums(static_cast<int64_t>(B) * Cout * 2);
    op_t* a0 = nullptr; op_t* xr = nullptr; float2* tab0 = nullptr;
    ConvArgs c0;
    c0.wpack = w0; c0.bias = c0b; c0.bias_b = dense_row >= 0 ? dense + dense_row : nullptr; c0.bias_b_stride = dense_stride;
    c0.B = B; c0.T = To; c0.F = Fo; c0.Cout = Cout; c0.out_h16 = h1; c0.sums = h1_sums;
    // the (scale, shift) table of GroupNorm_0 is needed by the on-load path and by every backward pass
    tab0 = norm_table(x1.sums, C1, x2 ? x2->sums : nullptr, C2, g0w, g0b, T, F);
    float2* stats0 = norm_stats(x1.sums);
    if (mode == 0) {
      // GroupNorm_0 + SiLU applied by Conv_0 on load, straight from the 16-bit copies of the residual stream
      c0.seg[0] = seg(x1.h16, C1, 9, tab0, Cin, 1); c0.n_seg = 1;
      if (x2) { c0.seg[1] = seg(x2->h16, C2, 9, tab0 + C1, Cin, 1); c0.n_seg = 2; }
    } else {
      // resampling blocks: one pass does GroupNorm_0 + SiLU + FIR up/down of h and the FIR of the raw shortcut operand
      a0 = alloc<op_t>(npx * Cin);
      xr = alloc<op_t>(npx * Cin);
      {
        const op_t* h1s = x1.h16; const op_t* h2s = x2 ? x2->h16 : nullptr;
        op([=](cudaStream_t s) { return launch_gn_resample16(h1s, C1, h2s, C2, tab0, B, T, F, mode, a0, xr, s); }, FDBM_OP_NORM);
      }
      c0.seg[0] = seg(a0, Cin, 9); c0.n_seg = 1;
    }
    conv_op(c0);
    release(a0); release(tab0);
    float2* tab1 = norm_table(h1_sums, Cout, nullptr, 0, g1w, g1b, To, Fo);
    float2* stats1 = norm_stats(h1_sums);
    Act out = new_act(Cout, To, Fo);
    {
      ConvArgs c;
      c.seg[0] = seg(h1, Cout, 9, tab1, Cout, 1); c.n_seg = 1;
      if (shortcut) {
        if (mode == 0) {
          c.seg[c.n_seg++] = seg(x1.h16, C1, 1);
          if (x2) c.seg[c.n_seg++] = seg(x2->h16, C2, 1);
        } else {
          c.seg[c.n_seg++] = seg(xr, Cin, 1);
        }
      }
      c.wpack = w1; c.bias = bias1;
      if (!shortcut) c.residual_h16 = x1.h16;
      c.scale = 0.70710678118654752f; c.B = B; c.T = To; c.F = Fo; c.Cout = Cout;
      c.out_h16 = out.h16; c.sums = out.sums;
      if (comb) { c.comb_pyr = comb->pyr; c.comb_w = comb->w; c.comb_b = comb->b; c.comb_C = comb->Cp; }
      conv_op(c);
    }
    release(h1); if (train()) release(h1_sums); release(tab1);
    release(xr);

    if (train()) {
      // ------------------------------------------------------------------ backward of the block (recorded, replayed in reverse)
      bgroup();
      fdbm_plan* plp = P;
      const int64_t pxo = static_cast<int64_t>(To) * Fo;
      const Act xa = x1; const Act xb = x2 ? *x2 : Act();
      op_t *t1 = T1, *t2 = T2, *t3 = T3, *t4 = T4, *t5 = T5;
      double* sA = site_sums(static_cast<int64_t>(B) * Cout);       // dL/d(out) column sums: Conv_1 (and Conv_2) bias gradients
      double* sA1 = site_sums(static_cast<int64_t>(B) * Cout);      // g_h1 column sums: Conv_0 bias and FiLM gradients
      double* S = site_sums(static_cast<int64_t>(B) * Cout * 2);    // GroupNorm_1 backward sums
      float* dd = d_dense;
      defer_col_sums(sA, Cout, o_c1b);
      if (o_c2b >= 0) defer_col_sums(sA, Cout, o_c2b);
      defer_gn_param(S, Cout, o_g1w, o_g1b);
      defer_col_sums(sA1, Cout, o_c0b, dense_row >= 0 ? dd + dense_row : nullptr, dense_stride);
      if (comb) {
        const CombineArgs cb = *comb; const float* og = out.grad;
        bop([=](cudaStream_t s) {
          return launch_combine_bwd(og, cb.pyr, cb.Cp, static_cast<int64_t>(B) * pxo, Cout, plp->cur_inv, plp->grads + cb.w_off, plp->grads + cb.b_off, s);
        });
      }
      {   // gs = dL/d(out) / sqrt(2) as a 16-bit operand; identity shortcut: x.grad += gs; bias gradients
        const float* og = out.grad; float* xg = shortcut ? nullptr : xa.grad;
        bop([=](cudaStream_t s) {
          if (int rc = plp->grad_ensure(og, s)) return rc;
          return launch_grad_prepare(og, B, pxo, Cout, 0.70710678118654752f, t1, xg, sA, s, xg && plp->grad_first(xg), true);
        });
      }
      if (shortcut) {
        if (mode == 0) {
          op_t* wd1 = pack_d(o_c2w, Cout, C1, 1, Cin, 0);
          dgrad_op(t1, Cout, 1, wd1, C1, To, Fo, nullptr, xa.grad);
          WgradCall w; w.dy = t1; w.dy_ld = Cout; w.Cout = Cout; w.x = xa.h16; w.x_ld = C1; w.Cin = C1; w.ksize = 1; w.T = To; w.F = Fo;
          w.Cin_total = Cin; w.ci_off = 0;
          wgrad_op(w, o_c2w);
          if (x2) {
            op_t* wd2 = pack_d(o_c2w, Cout, C2, 1, Cin, C1);
            dgrad_op(t1, Cout, 1, wd2, C2, To, Fo, nullptr, xb.grad);
            w.x = xb.h16; w.x_ld = C2; w.Cin = C2; w.ci_off = C1;
            wgrad_op(w, o_c2w);
          }
        } else {
          op_t* wd = pack_d(o_c2w, Cout, Cin, 1);
          dgrad_op(t1, Cout, 1, wd, Cin, To, Fo, t3, nullptr);
          float* xg = xa.grad;
          // adjoint of the FIR on the shortcut operand: adjoint(down) = up / 4, adjoint(up) = 4 * down
          bop([=](cudaStream_t s) {
            if (int rc = plp->grad_ensure(xg, s)) return rc;                 // this kernel only adds
            return launch_fir_resample16(t3, Cin, 0, B, To, Fo, Cin, mode == 1 ? 2 : 1, mode == 1 ? 0.25f : 4.0f, nullptr, xg, s);
          });
          WgradCall w; w.dy = t1; w.dy_ld = Cout; w.Cout = Cout; w.x = xr; w.x_ld = Cin; w.Cin = Cin; w.ksize = 1; w.T = To; w.F = Fo;
          wgrad_op(w, o_c2w);
        }
      }
      // Conv_1: wgrad needs a1 = SiLU(GroupNorm_1(h1)) (recomputed from the saved 16-bit h1), dgrad gives g_a1
      bop([=](cudaStream_t s) { return launch_groupnorm_act(h1, 1, h1_sums, Cout, nullptr, nullptr, 0, g1w, g1b, B, To, Fo, 1, 0, t2, nullptr, s); });
      { WgradCall w; w.dy = t1; w.dy_ld = Cout; w.Cout = Cout; w.x = t2; w.x_ld = Cout; w.Cin = Cout; w.ksize = 3; w.T = To; w.F = Fo; wgrad_op(w, o_c1w); }
      dgrad_op(t1, Cout, 9, pack_d(o_c1w, Cout, Cout, 3), Cout, To, Fo, t3, nullptr);
      bop([=](cudaStream_t s) {     // GroupNorm_1 backward: g_h1 (16-bit) + its per-(b,c) sums (Conv_0 bias and FiLM gradients)
        if (int rc = launch_gn_bwd_reduce(t3, Cout, 0, h1, 1, Cout, Cout, 0, tab1, stats1, 1, B, pxo, S, s)) return rc;
        return launch_gn_bwd_apply(t3, Cout, 0, h1, 1, Cout, Cout, 0, tab1, stats1, g1w, 1, B, pxo, S, nullptr, t4, sA1, s, false, true);
      });
      // Conv_0: a0 recomputed (or the saved resampled one), wgrad, dgrad, GroupNorm_0 backward into x.grad
      const op_t* a0b = a0;
      if (mode == 0) {
        const op_t* s1 = xa.h16; const double* q1 = xa.sums; const op_t* s2 = x2 ? xb.h16 : nullptr; const double* q2 = x2 ? xb.sums : nullptr;
        bop([=](cudaStream_t s) { return launch_groupnorm_act(s1, 1, q1, C1, s2, q2, C2, g0w, g0b, B, T, F, 1, 0, t2, nullptr, s); });
        a0b = t2;
      }
      { WgradCall w; w.dy = t4; w.dy_ld = Cout; w.Cout = Cout; w.x = a0b; w.x_ld = Cin; w.Cin = Cin; w.ksize = 3; w.T = To; w.F = Fo; wgrad_op(w, o_c0w); }
      dgrad_op(t4, Cout, 9, pack_d(o_c0w, Cout, Cin, 3), Cin, To, Fo, t3, nullptr);
      const op_t* g_act = t3;
      if (mode != 0) {
        bop([=](cudaStream_t s) { return launch_fir_resample16(t3, Cin, 0, B, To, Fo, Cin, mode == 1 ? 2 : 1, mode == 1 ? 0.25f : 4.0f, t5, nullptr, s); });
        g_act = t5;
      }
      gn_bwd(g_act, x1, x2, tab0, stats0, o_g0w, o_g0b, 1);
    }
    return out;
  }
  // AttnBlockpp (layerspp.py:75-91)
  Act attn(const Mod& m, const Act& x) {
    const int B = P->B, C = m.cin, T = x.T, F = x.F;
    const std::string p = pre(m);
    const int64_t o_gw = param(p + "GroupNorm_0.weight", C), o_gb = param(p + "GroupNorm_0.bias", C);
    const float* gw = pp(o_gw); const float* gb = pp(o_gb);
    // q, k, v projections as one GEMM with 3C outputs; biases are three consecutive slots
    const int64_t o_b0 = param(p + "NIN_0.b", C), o_b1 = param(p + "NIN_1.b", C), o_b2 = param(p + "NIN_2.b", C), o_b3 = param(p + "NIN_3.b", C);
    const float* bq = pp(o_b0);
    const float* b3 = pp(o_b3);
    const int64_t o_w0 = param(p + "NIN_0.W", static_cast<int64_t>(C) * C), o_w1 = param(p + "NIN_1.W", static_cast<int64_t>(C) * C),
                  o_w2 = param(p + "NIN_2.W", static_cast<int64_t>(C) * C), o_w3 = param(p + "NIN_3.W", static_cast<int64_t>(C) * C);
    op_t* wqkv = pack(p + "NIN_0.W", C, -1, "", 0, C, 3 * C, 0);
    pack(p + "NIN_1.W", C, -1, "", 0, C, 3 * C, C, wqkv);
    pack(p + "NIN_2.W", C, -1, "", 0, C, 3 * C, 2 * C, wqkv);
    op_t* w3 = pack(p + "NIN_3.W", C, -1, "", 0, C);
    const int64_t npx = static_cast<int64_t>(B) * T * F;
    float2* tab = norm_table(x.sums, C, nullptr, 0, gw, gb, T, F);
    float2* stats = norm_stats(x.sums);
    op_t* qkv = alloc<op_t>(npx * 3 * C);
    {
      ConvArgs c;
      c.seg[0] = seg(x.h16, C, 1, tab, C, 0); c.n_seg = 1;      // GroupNorm_0 (no activation) on load
      c.wpack = wqkv; c.bias = bq; c.B = B; c.T = T; c.F = F; c.Cout = 3 * C;
      c.out_h16 = qkv;
      conv_op(c);
    }
    release(tab);
    op_t* o = alloc<op_t>(npx * C);
    const int fp32_probs = train() ? 1 : 0;
    op([=](cudaStream_t s) { return launch_attention(qkv, qkv + C, qkv + 2 * C, 3 * C, B, T * F, C, o, C, s, fp32_probs); }, FDBM_OP_ATTN);
    release(qkv);
    Act out = new_act(C, T, F);
    {
      ConvArgs c;
      c.seg[0] = seg(o, C, 1); c.n_seg = 1;
      c.wpack = w3; c.bias = b3; c.scale = 0.70710678118654752f;
      c.residual_h16 = x.h16;
      c.B = B; c.T = T; c.F = F; c.Cout = C; c.out_h16 = out.h16; c.sums = out.sums;
      conv_op(c);
    }
    release(o);
    if (train()) {
      bgroup();
      fdbm_plan* plp = P;
      const int64_t px = static_cast<int64_t>(T) * F;
      op_t *t1 = T1, *t2 = T2, *t3 = T3, *t4 = T4;
      double* sA = site_sums(static_cast<int64_t>(B) * C); float* asc = att_scratch;
      double* sQ[3] = {site_sums(static_cast<int64_t>(B) * C), site_sums(static_cast<int64_t>(B) * C), site_sums(static_cast<int64_t>(B) * C)};
      defer_col_sums(sA, C, o_b3);
      const Act xa = x;
      { const float* og = out.grad; float* xg = xa.grad;
        bop([=](cudaStream_t s) {
          if (int rc = plp->grad_ensure(og, s)) return rc;
          return launch_grad_prepare(og, B, px, C, 0.70710678118654752f, t1, xg, sA, s, plp->grad_first(xg), true);
        }); }
      { WgradCall w; w.dy = t1; w.dy_ld = C; w.Cout = C; w.x = o; w.x_ld = C; w.Cin = C; w.ksize = 1; w.T = T; w.F = F; w.layout = 1; wgrad_op(w, o_w3); }
      dgrad_op(t1, C, 1, pack_d(o_w3, C, C, -1), C, T, F, t3, nullptr);
      const int64_t o_b[3] = {o_b0, o_b1, o_b2};
      for (int i = 0; i < 3; ++i) defer_col_sums(sQ[i], C, o_b[i]);
      double *sq0 = sQ[0], *sq1 = sQ[1], *sq2 = sQ[2];
      bop([=](cudaStream_t s) {
        if (int rc = launch_attention_bwd(qkv, B, T * F, C, t3, asc, t4, s)) return rc;
        double* const sq[3] = {sq0, sq1, sq2};
        for (int i = 0; i < 3; ++i)
          if (int rc = launch_col_sums16(t4, 3 * C, i * C, B, px, C, sq[i], s, true)) return rc;
        return FDBM_OK;
      });
      { const op_t* s1 = xa.h16; const double* q1 = xa.sums;
        bop([=](cudaStream_t s) { return launch_groupnorm_act(s1, 1, q1, C, nullptr, nullptr, 0, gw, gb, B, T, F, 0, 0, t2, nullptr, s); }); }
      const int64_t o_w[3] = {o_w0, o_w1, o_w2};
      for (int i = 0; i < 3; ++i) {
        WgradCall w; w.dy = t4; w.dy_ld = 3 * C; w.dy_coff = i * C; w.Cout = C; w.x = t2; w.x_ld = C; w.Cin = C; w.ksize = 1; w.T = T; w.F = F; w.layout = 1;
        wgrad_op(w, o_w[i]);
      }
      // dgrad of the fused q|k|v projection: K = 3C over the three transposed NIN matrices
      op_t* wd = pack_d(o_w0, C, C, -1);
      pack_d(o_w1, C, C, -1); pack_d(o_w2, C, C, -1);          // consecutive regions: K blocks q, k, v
      dgrad_op(t4, 3 * C, 1, wd, C, T, F, t3, nullptr);
      gn_bwd(t3, x, nullptr, tab, stats, o_gw, o_gb, 0);
    }
    return out;
  }

  int build() {
    fdbm_plan& pl = *P;
    const fdbm_arch& A = pl.arch;
    const int B = pl.B, nf = A.nf, Cp = pl.Cin, L = A.n_levels;
    size_t mi = 0;
    auto next = [&]() -> const Mod& { return pl.mods[mi++]; };
    wp_off = 0; dense_off = 0; wd_off = 0; ws_need = 0; groups.clear();
    sums_used = 0;
    if (!dry && P->sums_pool_bytes > 0) {
      sums_pool = alloc<uint8_t>(P->sums_pool_bytes);
      uint8_t* pool = sums_pool; const int64_t pool_bytes = P->sums_pool_bytes;
      op([=](cudaStream_t s) { FDBM_CUDA(cudaMemsetAsync(pool, 0, pool_bytes, s)); return FDBM_OK; }, FDBM_OP_STATS);
    }
    if (train()) {
      // shared backward scratch: the largest 16-bit operand of the network is [B, T, F, 2 nf] at level 0
      const int64_t big = static_cast<int64_t>(B) * pl.T * pl.F * 2 * nf;
      T1 = alloc<op_t>(big); T2 = alloc<op_t>(big); T3 = alloc<op_t>(big); T4 = alloc<op_t>(big); T5 = alloc<op_t>(big);
      Sbuf = alloc<double>(static_cast<int64_t>(B) * 1024 * 2);
      sumsA = alloc<double>(static_cast<int64_t>(B) * 1024);
      const int Lmax = (pl.T >> 4) * (pl.F >> 4);                     // attention runs at the 16-bin level
      att_scratch = alloc<float>(2ll * B * Lmax * Lmax);
      zero_bias = pp(derived(1024));
    }

    // ---- time embedding + all Dense_0 projections (one table [B, dense_rows])
    float* temb_act = nullptr; float* dense = nullptr;
    if (!A.predictive) {
      const Mod& mf = next(); const Mod& l1 = next(); const Mod& l2 = next();
      const float* fw = pp(param(pre(mf) + "W", nf));
      const int64_t o_w1 = param(pre(l1) + "weight", static_cast<int64_t>(4 * nf) * 2 * nf), o_b1 = param(pre(l1) + "bias", 4 * nf);
      const int64_t o_w2 = param(pre(l2) + "weight", static_cast<int64_t>(4 * nf) * 4 * nf), o_b2 = param(pre(l2) + "bias", 4 * nf);
      const float* w1 = pp(o_w1); const float* b1 = pp(o_b1); const float* w2 = pp(o_w2); const float* b2 = pp(o_b2);
      // Dense_0 weights / biases of all residual blocks, contiguous and in execution order
      int rows = 0; int64_t dw0 = -1, db0 = -1;
      for (const Mod& m : pl.mods) if (m.kind == Mod::RES) {
        const int64_t o = param(pre(m) + "Dense_0.weight", static_cast<int64_t>(m.cout) * 4 * nf);
        if (dw0 < 0) dw0 = o;
        rows += m.cout;
      }
      for (const Mod& m : pl.mods) if (m.kind == Mod::RES) {
        const int64_t o = param(pre(m) + "Dense_0.bias", m.cout);
        if (db0 < 0) db0 = o;
      }
      pl.dense_rows = rows;
      temb_act = alloc<float>(static_cast<int64_t>(B) * 4 * nf);
      dense = alloc<float>(static_cast<int64_t>(B) * rows);
      const float* dwp = pp(dw0); const float* dbp = pp(db0);
      fdbm_plan* plp = P;
      // the sampler passes one time for the whole batch (stride 0): one embedding row, read by every utterance
      op([=](cudaStream_t s) {
        return launch_temb(plp->cur_t, fw, nf, w1, b1, w2, b2, plp->cur_t_stride == 0 ? 1 : B, plp->cur_t_stride, temb_act, s);
      }, FDBM_OP_SMALL);
      op([=](cudaStream_t s) { return launch_dense_all(temb_act, dwp, dbp, plp->cur_t_stride == 0 ? 1 : B, 4 * nf, rows, dense, s); }, FDBM_OP_SMALL);
      if (train()) {
        // first group = last to run in backward: by then every block has left its FiLM gradient in d_dense
        d_dense = alloc<float>(static_cast<int64_t>(B) * rows);
        g_temb = alloc<float>(static_cast<int64_t>(B) * 4 * nf);
        float* dd = d_dense; float* gt = g_temb;
        bgroup();
        bop([=](cudaStream_t s) {
          // last group of the backward: every site has left its sums; reduce them into the parameter gradients (and the FiLM
          // rows of d_dense that the time-embedding backward below consumes) in one launch
          if (int rc = launch_deferred_sums(plp->defer_descs_d, static_cast<int>(plp->defer_descs.size()), plp->cur_inv, s)) return rc;
          return launch_dense_temb_bwd(dd, temb_act, dwp, B, 4 * nf, rows, plp->grads + dw0, plp->grads + db0, gt, plp->cur_t, fw, nf, w1, b1, w2,
                                       b2, plp->cur_t_stride, plp->grads + o_w1, plp->grads + o_b1, plp->grads + o_w2, plp->grads + o_b2, s);
        });
      }
    }
    const int dstride = pl.dense_rows;

    // ---- input packing and first convolution
    int T = pl.T, F = pl.F;
    float* pyr_in = alloc<float>(static_cast<int64_t>(B) * T * F * Cp);
    {
      fdbm_plan* plp = P; const int Tc = T, Fc = F; float* dst = pyr_in; const bool pred = A.predictive;
      op([=](cudaStream_t s) { return launch_pack_input(plp->cur_x, pred ? nullptr : plp->cur_y, B, Tc, plp->F_io, Fc, Cp, dst, s); }, FDBM_OP_SKINNY);
    }
    std::vector<Act> hs;
    {
      const Mod& m = next();
      const int64_t o_w = param(pre(m) + "weight", static_cast<int64_t>(nf) * Cp * 9), o_b = param(pre(m) + "bias", nf);
      const float* w = pp(o_w); const float* b = pp(o_b);
      // first conv (4 -> nf, 3x3) on the tensor cores: im2col to one 64-wide K-block, then a K=64 GEMM
      op_t* wp = reinterpret_cast<op_t*>(reinterpret_cast<uint8_t*>(P->wpacked) + wp_off);
      wp_off += (static_cast<int64_t>(nf) * 64 * 2 + 1023) / 1024 * 1024;
      pack_op([=](cudaStream_t s) { return launch_pack_conv_weights(w, Cp, -2, nullptr, 0, nf, nf, 0, wp, s); });
      Act h0 = new_act(nf, T, F);
      const int Tc = T, Fc = F; float* src = pyr_in;
      op_t* cols = alloc<op_t>(static_cast<int64_t>(B) * T * F * 64);
      op([=](cudaStream_t s) { return launch_im2col_input(src, Cp, B, Tc, Fc, cols, s); }, FDBM_OP_SKINNY);
      ConvArgs c;
      c.seg[0] = seg(cols, 64, 1); c.n_seg = 1;
      c.wpack = wp; c.bias = b; c.B = B; c.T = T; c.F = F; c.Cout = nf;
      c.out_h16 = h0.h16; c.sums = h0.sums;
      conv_op(c, 2.0 * B * T * F * nf * 9.0 * Cp);
      release(cols);
      if (train()) {
        bgroup();
        fdbm_plan* plp = P; op_t* t1 = T1; double* sA = site_sums(static_cast<int64_t>(B) * nf); const float* g0 = h0.grad;
        defer_col_sums(sA, nf, o_b);
        const int64_t px = static_cast<int64_t>(T) * F;
        bop([=](cudaStream_t s) {
          if (int rc = plp->grad_ensure(g0, s)) return rc;
          return launch_grad_prepare(g0, B, px, nf, 1.0f, t1, nullptr, sA, s, false, true);
        });
        WgradCall wc; wc.dy = t1; wc.dy_ld = nf; wc.Cout = nf; wc.x = cols; wc.x_ld = 64; wc.Cin = 64; wc.ksize = 1; wc.T = T; wc.F = F;
        wc.layout = 2; wc.aux = Cp;
        wgrad_op(wc, o_w);
      }
      hs.push_back(h0);
    }
    // ---- down path
    for (int lvl = 0; lvl < L; ++lvl) {
      for (int blk = 0; blk < A.num_res_blocks; ++blk) {
        Act h = resblock(next(), hs.back(), nullptr, dense, dstride);
        if (h.F == A.attn_resolution) { Act h2 = attn(next(), h); free_act(h); h = h2; }
        hs.push_back(h);
      }
      if (lvl != L - 1) {
        // input pyramid one level down, then the down-sampling block whose Conv_1 epilogue also applies the
        // Combine (layerspp.py:52-59): h = resblock(...) + conv1x1(4 -> C)(pyramid)
        const Mod& mr = next();
        float* pyr_next = alloc<float>(static_cast<int64_t>(B) * (T / 2) * (F / 2) * Cp);
        {
          const int Tc = T, Fc = F; float* src = pyr_in;
          op([=](cudaStream_t s) { return launch_fir_resample(src, B, Tc, Fc, Cp, 1, pyr_next, s); }, FDBM_OP_SKINNY);
        }
        release(pyr_in);
        pyr_in = pyr_next;
        const Mod& m = pl.mods[mi];               // the Combine module follows the block
        CombineArgs cb;
        cb.pyr = pyr_in; cb.Cp = Cp;
        cb.w_off = param(pre(m) + "Conv_0.weight", static_cast<int64_t>(m.cout) * Cp); cb.b_off = param(pre(m) + "Conv_0.bias", m.cout);
        cb.w = pp(cb.w_off); cb.b = pp(cb.b_off);
        Act h = resblock(mr, hs.back(), nullptr, dense, dstride, &cb);
        next();
        T /= 2; F /= 2;
        hs.push_back(h);
      }
    }
    release(pyr_in);
    // ---- bottleneck
    Act h = hs.back();                      // still owned by the skip stack
    {
      Act a = resblock(next(), h, nullptr, dense, dstride);
      Act b2 = attn(next(), a); free_act(a);
      Act c = resblock(next(), b2, nullptr, dense, dstride); free_act(b2);
      h = c;
    }
    // ---- up path
    float* pyramid = nullptr;
    float* gpyr = nullptr;                   // training: gradient buffer of the current pyramid level
    for (int lvl = L - 1; lvl >= 0; --lvl) {
      for (int blk = 0; blk < A.num_res_blocks + 1; ++blk) {
        Act skip = hs.back(); hs.pop_back();
        Act o = resblock(next(), h, &skip, dense, dstride);
        free_act(h); free_act(skip);
        h = o;
      }
      if (h.F == A.attn_resolution) { Act h2 = attn(next(), h); free_act(h); h = h2; }
      {
        const Mod& mg = next(); const Mod& mc = next();
        const int C = mg.cin, Tc = h.T, Fc = h.F;
        const int64_t o_gw = param(pre(mg) + "weight", C), o_gb = param(pre(mg) + "bias", C);
        const int64_t o_w = param(pre(mc) + "weight", static_cast<int64_t>(Cp) * C * 9), o_b = param(pre(mc) + "bias", Cp);
        const float* gw = pp(o_gw); const float* gb = pp(o_gb);
        const float* w = pp(o_w); const float* b = pp(o_b);
        // C -> 4 conv on the tensor cores: weight rows padded with zeros to the narrowest MMA N (16)
        op_t* wp = reinterpret_cast<op_t*>(reinterpret_cast<uint8_t*>(P->wpacked) + wp_off);
        const int64_t wbytes = conv_wpack_bytes(C, 3, 0, 16);
        wp_off += (wbytes + 1023) / 1024 * 1024;
        pack_op([=](cudaStream_t s) {
          FDBM_CUDA(cudaMemsetAsync(wp, 0, wbytes, s));
          return launch_pack_conv_weights(w, C, 3, nullptr, 0, Cp, 16, 0, wp, s);
        });
        float* pyr_new = alloc<float>(static_cast<int64_t>(B) * Tc * Fc * Cp);
        float* prev = pyramid;
        float2* tab = norm_table(h.sums, C, nullptr, 0, gw, gb, Tc, Fc);
        float2* stats = norm_stats(h.sums);
        ConvArgs c;
        c.seg[0] = seg(h.h16, C, 9, tab, C, 1); c.n_seg = 1;     // GroupNorm + SiLU on load
        c.wpack = wp; c.bias = b; c.B = B; c.T = Tc; c.F = Fc; c.Cout = 16; c.narrow_n = true;
        c.pyr_out = pyr_new; c.pyr_prev = prev; c.pyr_C = Cp;
        conv_op(c, 2.0 * B * Tc * Fc * Cp * 9.0 * C);
        release(tab);
        if (train()) {
          // progressive output backward (ncsnpp_v2.py:338-359): g_pyr of this level arrives from the finer level (or from
          // the output layer); the coarser level receives adjoint(FIR up) = 4 * FIR down of it
          float* g_new = alloc<float>(static_cast<int64_t>(B) * Tc * Fc * Cp);
          float* g_prev = gpyr;
          gpyr = g_new;
          bgroup();
          fdbm_plan* plp = P; op_t *t1 = T1, *t2 = T2, *t3 = T3;
          const int64_t px = static_cast<int64_t>(Tc) * Fc;
          op_t* wd = reinterpret_cast<op_t*>(reinterpret_cast<uint8_t*>(P->wpacked_d) + wd_off);
          wd_off += (static_cast<int64_t>(C) * 64 * 2 + 1023) / 1024 * 1024;
          pack_op([=](cudaStream_t s) { return launch_pack_pyr_dgrad(w, C, Cp, wd, s); });
          bop([=](cudaStream_t s) {
            if (g_prev) if (int rc = launch_fir_resample_scaled(g_new, B, Tc, Fc, Cp, 1, 4.0f, g_prev, s)) return rc;
            if (int rc = launch_small_col_sums(g_new, static_cast<int64_t>(B) * px, Cp, plp->cur_inv, plp->grads + o_b, s)) return rc;
            return launch_im2col_input(g_new, Cp, B, Tc, Fc, t1, s);
          });
          dgrad_op(t1, 64, 1, wd, C, Tc, Fc, t3, nullptr);
          { const op_t* s1 = h.h16; const double* q1 = h.sums;
            bop([=](cudaStream_t s) { return launch_groupnorm_act(s1, 1, q1, C, nullptr, nullptr, 0, gw, gb, B, Tc, Fc, 1, 0, t2, nullptr, s); }); }
          WgradCall wc; wc.dy = t2; wc.dy_ld = C; wc.Cout = C; wc.x = t1; wc.x_ld = 64; wc.Cin = 64; wc.ksize = 1; wc.T = Tc; wc.F = Fc;
          wc.layout = 3; wc.aux = Cp;
          wgrad_op(wc, o_w);
          gn_bwd(t3, h, nullptr, tab, stats, o_gw, o_gb, 1);
        }
        release(pyramid);
        pyramid = pyr_new;
      }
      if (lvl != 0) { Act o = resblock(next(), h, nullptr, dense, dstride); free_act(h); h = o; }
    }
    free_act(h);
    if (mi != pl.mods.size() || !hs.empty()) { set_error("plan: module walk out of sync (%zu of %zu)", mi, pl.mods.size()); return FDBM_EINVAL; }
    {
      const int64_t o_w = param("output_layer.weight", 2 * Cp), o_b = param("output_layer.bias", 2);
      const float* w = pp(o_w); const float* b = pp(o_b);
      const int Tc = pl.T, Fc = pl.F; fdbm_plan* plp = P; float* pyr = pyramid;
      op([=](cudaStream_t s) { return launch_output_layer(pyr, Cp, w, b, B, Tc, Fc, plp->F_io, plp->cur_out, s); }, FDBM_OP_SKINNY);
      if (train()) {
        bgroup();
        float* g0 = gpyr;
        bop([=](cudaStream_t s) {
          return launch_output_layer_bwd(plp->cur_gout, pyr, Cp, w, B, Tc, Fc, plp->F_io, plp->cur_inv, g0, plp->grads + o_w, plp->grads + o_b, s);
        });
      }
    }
    release(pyramid);
    if (train() && !dry) {
      for (auto g = groups.rbegin(); g != groups.rend(); ++g)
        for (auto& f : *g) { P->bwd_ops.push_back(std::move(f.first)); P->bwd_kind.push_back(f.second); }
    }
    return FDBM_OK;
  }
};

int run_ops(fdbm_plan* plan, cudaStream_t s) {
  PdlBatchScope pdl(plan->train ? std::min(std::max(plan->B, 8), 32) : 8);   // training plans: short launches at every level (api.cu)
  for (auto& f : plan->ops) if (int rc = f(s)) return rc;
  return FDBM_OK;
}

}  // namespace

static int plan_create_impl(const fdbm_arch* arch, int batch, int n_frames, bool train, fdbm_plan** out) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(arch && out, "fdbm_plan_create: null pointer");
  FDBM_REQUIRE(batch > 0 && n_frames > 0, "fdbm_plan_create: batch and n_frames must be positive");
  FDBM_REQUIRE(arch->n_levels >= 1 && arch->n_levels <= 8, "fdbm_plan_create: n_levels out of range");
  FDBM_REQUIRE(arch->nf % 64 == 0 && arch->nf >= 64, "fdbm_plan_create: nf must be a multiple of 64 (got %d); the nf = 96 variants need 32-channel K-blocks", arch->nf);
  FDBM_REQUIRE(arch->image_size == 256, "fdbm_plan_create: image_size must be 256 (n_fft = 512 with the Nyquist bin dropped)");
  const int down = 1 << (arch->n_levels - 1);
  FDBM_REQUIRE(n_frames % down == 0, "fdbm_plan_create: n_frames %d must be a multiple of %d (pad_spec pads to 64)", n_frames, down);
  for (int i = 0; i < arch->n_levels; ++i) {
    const int c = arch->nf * arch->ch_mult[i];
    FDBM_REQUIRE(c == 64 || c % 128 == 0, "fdbm_plan_create: level %d has %d channels; supported: 64 or a multiple of 128", i, c);
  }
  FDBM_REQUIRE(arch->channel_block_real == 0 || (arch->channel_block_real == 96 && arch->nf == 128 && !train),
               "fdbm_plan_create: channel_block_real must be 0, or 96 with nf = 128 on an inference plan (got %d, nf %d)",
               arch->channel_block_real, arch->nf);
  FDBM_REQUIRE(!train || arch->nf >= 128, "fdbm_plan_create_train: the training step is built for nf >= 128");

  fdbm_plan* P = new fdbm_plan();
  P->arch = *arch; P->B = batch; P->T = n_frames; P->F = arch->image_size; P->F_io = arch->image_size + 1;
  P->Cin = arch->predictive ? 2 : 4;
  P->train = train;
  P->device = current_device();
  P->mods = build_modules(*arch);
  auto fail = [&](int rc) { fdbm_plan_destroy(P); return rc; };

  // pass 1 (dry): sizes.  A 1 TiB virtual arena never fails; its peak is the real requirement.
  Builder b1{P};
  b1.dry = true;
  P->arena = reinterpret_cast<uint8_t*>(uintptr_t(1) << 30);      // fake non-null base for the sizing pass
  b1.arena.reset(int64_t(1) << 40);
  if (int rc = b1.build()) return fail(rc);
  P->sums_pool_bytes = b1.sums_used;
  P->defer_pool_bytes = b1.defer_used;
  P->arena_bytes = b1.arena.peak() + (P->sums_pool_bytes + 1023) / 1024 * 1024;
  P->arena = nullptr;
  P->wpacked_bytes = b1.wp_off;
  P->wpacked_d_bytes = b1.wd_off;
  P->wgrad_ws_bytes = b1.ws_need;
  const int64_t params_numel = P->params_numel;
  // d_buf for the sampler
  const int64_t spec_elems = static_cast<int64_t>(batch) * P->F_io * n_frames * 2;
  cudaError_t e;
  if ((e = cudaMalloc(&P->arena, P->arena_bytes)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(arena)", __FILE__, __LINE__));
  if ((e = cudaMalloc(&P->params, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(params)", __FILE__, __LINE__));
  if ((e = cudaMalloc(&P->wpacked, P->wpacked_bytes)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(wpacked)", __FILE__, __LINE__));
  if ((e = cudaMalloc(&P->d_buf, spec_elems * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(d_buf)", __FILE__, __LINE__));
  if ((e = cudaMemset(P->params, 0, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset", __FILE__, __LINE__));
  P->extra_bytes = spec_elems * sizeof(float);
  if (train) {
    if ((e = cudaMalloc(&P->grads, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(grads)", __FILE__, __LINE__));
    if (P->defer_pool_bytes && (e = cudaMalloc(&P->defer_pool, P->defer_pool_bytes)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(deferred sums pool)", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->wpacked_d, std::max<int64_t>(P->wpacked_d_bytes, 1024))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(wpacked_d)", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->wgrad_ws, std::max<int64_t>(P->wgrad_ws_bytes, 1024))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(wgrad_ws)", __FILE__, __LINE__));
    if ((e = cudaMemset(P->grads, 0, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset", __FILE__, __LINE__));
    // optimiser state: Adam moments, EMA shadow + the backup the evaluation swap parks the live parameters in
    float** bufs[4] = {&P->adam_m, &P->adam_v, &P->ema, &P->ema_backup};
    for (float** b : bufs) {
      if ((e = cudaMalloc(b, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(optimiser)", __FILE__, __LINE__));
      if ((e = cudaMemset(*b, 0, params_numel * sizeof(float))) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset", __FILE__, __LINE__));
    }
    if ((e = cudaMalloc(&P->opt_scratch, 1025 * sizeof(double))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(opt_scratch)", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->opt_state, 4 * sizeof(double))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(opt_state)", __FILE__, __LINE__));
    if ((e = cudaMemset(P->opt_state, 0, 4 * sizeof(double))) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset", __FILE__, __LINE__));
    P->extra_bytes += P->defer_pool_bytes + params_numel * 4 * 5 + std::max<int64_t>(P->wpacked_d_bytes, 1024) + std::max<int64_t>(P->wgrad_ws_bytes, 1024);
  } else if (!arch->predictive) {
    // sampler staging: the graph of the N-step loop reads y / x / times / coefficients / seed from these fixed buffers
    const size_t spec_bytes = spec_elems * sizeof(float);
    if ((e = cudaMalloc(&P->smp_y, spec_bytes)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(sampler y)", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->smp_x, spec_bytes)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(sampler x)", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->smp_times, sizeof(float) * fdbm_plan::kMaxSteps)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->smp_coef, sizeof(float) * 3 * fdbm_plan::kMaxSteps)) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc", __FILE__, __LINE__));
    if ((e = cudaMalloc(&P->smp_rng, 2 * sizeof(uint64_t))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc", __FILE__, __LINE__));
    if ((e = cudaMallocHost(&P->smp_pinned, kSlotBytes * fdbm_plan::kRing)) != cudaSuccess) return fail(cuda_fail(e, "cudaMallocHost", __FILE__, __LINE__));
    for (int i = 0; i < fdbm_plan::kRing; ++i)
      if ((e = cudaEventCreateWithFlags(&P->smp_ev[i], cudaEventDisableTiming)) != cudaSuccess) return fail(cuda_fail(e, "cudaEventCreate", __FILE__, __LINE__));
    if ((e = cudaStreamCreateWithFlags(&P->capture_stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(cuda_fail(e, "cudaStreamCreate", __FILE__, __LINE__));
    P->extra_bytes += 2 * spec_bytes + sizeof(float) * 4 * fdbm_plan::kMaxSteps + 16;
  }

  // pass 2: identical walk, now recording launches against real addresses
  P->params_numel = 0;
  P->slots.clear();
  Builder b2{P};
  b2.dry = false;
  b2.arena.reset(P->arena_bytes);
  if (int rc = b2.build()) return fail(rc);
  P->n_bwd_launches = static_cast<int>(P->bwd_ops.size());
  if (!P->defer_descs.empty()) {
    if ((e = cudaMalloc(&P->defer_descs_d, P->defer_descs.size() * sizeof(DeferDesc))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(deferred sums)", __FILE__, __LINE__));
    if ((e = cudaMemcpy(P->defer_descs_d, P->defer_descs.data(), P->defer_descs.size() * sizeof(DeferDesc), cudaMemcpyHostToDevice)) != cudaSuccess)
      return fail(cuda_fail(e, "cudaMemcpy(deferred sums)", __FILE__, __LINE__));
  }
  if (b2.defer_used != P->defer_pool_bytes) { set_error("plan: deferred-sums pool diverged from the sizing pass"); return fail(FDBM_EINVAL); }
  if (!P->pack_descs.empty()) {
    long long nb = 0;
    for (auto& d : P->pack_descs) { d.first_block = nb; nb += (d.total + kPackChunk - 1) / kPackChunk; }
    P->pack_blocks = nb;
    if ((e = cudaMalloc(&P->pack_descs_d, P->pack_descs.size() * sizeof(PackDesc))) != cudaSuccess) return fail(cuda_fail(e, "cudaMalloc(pack descriptors)", __FILE__, __LINE__));
    if ((e = cudaMemcpy(P->pack_descs_d, P->pack_descs.data(), P->pack_descs.size() * sizeof(PackDesc), cudaMemcpyHostToDevice)) != cudaSuccess)
      return fail(cuda_fail(e, "cudaMemcpy(pack descriptors)", __FILE__, __LINE__));
  }
  if (P->params_numel != params_numel || b2.wp_off != P->wpacked_bytes || b2.wd_off != P->wpacked_d_bytes) {
    set_error("plan: second pass diverged from the sizing pass");
    return fail(FDBM_EINVAL);
  }
  *out = P;
  return FDBM_OK;
}

// packed 16-bit weights (forward and dgrad) <- the flat fp32 parameter buffer
static int run_pack_ops(fdbm_plan* plan, cudaStream_t s) {
  if (int rc = launch_pack_batch(plan->pack_descs_d, static_cast<int>(plan->pack_descs.size()), plan->pack_blocks, s)) return rc;
  for (auto& f : plan->pack_ops) if (int rc = f(s)) return rc;
  return FDBM_OK;
}

extern "C" int fdbm_plan_create(const fdbm_arch* arch, int batch, int n_frames, fdbm_plan** out) {
  return plan_create_impl(arch, batch, n_frames, false, out);
}

extern "C" int fdbm_plan_create_train(const fdbm_arch* arch, int batch, int n_frames, fdbm_plan** out) {
  FDBM_REQUIRE(arch && !arch->predictive, "fdbm_plan_create_train: the training step is built for the bridge backbone (predictive = 0)");
  return plan_create_impl(arch, batch, n_frames, true, out);
}

// dL/dparams of the last fdbm_ncsnpp_forward on a training plan.  g_out = loss_scale * dL/dD, cplx [B,1,257,T].
extern "C" int fdbm_ncsnpp_backward(fdbm_plan* plan, const float* g_out, float loss_scale, int accumulate, void* stream) {
  FDBM_REQUIRE(plan && g_out && loss_scale > 0.f, "fdbm_ncsnpp_backward: bad arguments");
  if (int rc = plan_guard(plan, "fdbm_ncsnpp_backward")) return rc;
  if (!plan->train) { set_error("fdbm_ncsnpp_backward: not a training plan (use fdbm_plan_create_train)"); return FDBM_ESTATE; }
  if (!plan->weights_ready || !plan->cur_x) { set_error("fdbm_ncsnpp_backward: no forward pass to differentiate"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  plan->cur_gout = g_out; plan->cur_inv = 1.0f / loss_scale;
  if (!accumulate) FDBM_CUDA(cudaMemsetAsync(plan->grads, 0, plan->params_numel * sizeof(float), s));
  if (plan->defer_pool_bytes) FDBM_CUDA(cudaMemsetAsync(plan->defer_pool, 0, plan->defer_pool_bytes, s));
  plan->grads_begin();
  PdlBatchScope pdl(std::min(std::max(plan->B, 8), 32));
  for (auto& f : plan->bwd_ops) if (int rc = f(s)) return rc;
  return FDBM_OK;
}

// measurement aid: the backward of the last forward, one CUDA event pair per recorded op (an op may be 1-5 launches)
extern "C" int fdbm_plan_profile_backward(fdbm_plan* plan, const float* g_out, float loss_scale, float* ms, int* kinds, int max_ops,
                                          void* stream) {
  FDBM_REQUIRE(plan && g_out && ms && kinds && plan->train, "fdbm_plan_profile_backward: bad arguments");
  if (int rc = plan_guard(plan, "fdbm_plan_profile_backward")) return rc;
  const int n = static_cast<int>(plan->bwd_ops.size());
  FDBM_REQUIRE(max_ops >= n, "fdbm_plan_profile_backward: need room for %d entries", n);
  cudaStream_t s = as_stream(stream);
  plan->cur_gout = g_out; plan->cur_inv = 1.0f / loss_scale;
  FDBM_CUDA(cudaMemsetAsync(plan->grads, 0, plan->params_numel * sizeof(float), s));
  if (plan->defer_pool_bytes) FDBM_CUDA(cudaMemsetAsync(plan->defer_pool, 0, plan->defer_pool_bytes, s));
  plan->grads_begin();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) FDBM_CUDA(cudaEventCreate(&e));
  int rc = FDBM_OK;
  FDBM_CUDA(cudaEventRecord(ev[0], s));
  for (int i = 0; i < n && rc == FDBM_OK; ++i) {
    rc = plan->bwd_ops[i](s);
    if (rc == FDBM_OK && cudaEventRecord(ev[i + 1], s) != cudaSuccess) rc = FDBM_ECUDA;
  }
  if (rc == FDBM_OK && cudaStreamSynchronize(s) != cudaSuccess) rc = cuda_fail(cudaGetLastError(), "cudaStreamSynchronize", __FILE__, __LINE__);
  for (int i = 0; i < n && rc == FDBM_OK; ++i) { cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]); kinds[i] = plan->bwd_kind[i]; }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc == FDBM_OK ? n : rc;
}

extern "C" int fdbm_plan_param_info(const fdbm_plan* plan, const char* name, int64_t* offset, int64_t* numel) {
  FDBM_REQUIRE(plan && name, "fdbm_plan_param_info: null pointer");
  auto it = plan->slots.find(name);
  FDBM_REQUIRE(it != plan->slots.end(), "fdbm_plan_param_info: unknown tensor '%s'", name);
  if (offset) *offset = it->second.off;
  if (numel) *numel = it->second.numel;
  return FDBM_OK;
}

extern "C" int fdbm_plan_buffers(fdbm_plan* plan, float** params, float** grads, float** ema, int64_t* numel) {
  FDBM_REQUIRE(plan, "fdbm_plan_buffers: null plan");
  if (params) *params = plan->params;
  if (grads) *grads = plan->grads;
  if (ema) *ema = plan->ema;
  if (numel) *numel = plan->params_numel;
  return FDBM_OK;
}

// re-derive the packed 16-bit weights (forward and dgrad packs) from the flat fp32 parameter buffer, e.g. after the caller
// has written it directly (DDP parameter broadcast from rank 0, checkpoint restore)
extern "C" int fdbm_plan_repack_weights(fdbm_plan* plan, void* stream) {
  if (int rc = plan_guard(plan, "fdbm_plan_repack_weights")) return rc;
  if (!plan->weights_ready) { set_error("fdbm_plan_repack_weights: weights not loaded"); return FDBM_ESTATE; }
  if (int rc = run_pack_ops(plan, as_stream(stream))) return rc;
  return FDBM_OK;
}

extern "C" int fdbm_plan_num_backward_launches(const fdbm_plan* plan) { return plan ? plan->n_bwd_launches : 0; }

// Adam + clip + EMA on the flat buffers, then the packed 16-bit weights are rebuilt from the updated parameters.
extern "C" int fdbm_plan_optimizer_step(fdbm_plan* plan, float grad_div, float clip_norm, float lr, float beta1, float beta2,
                                        float eps, int step, float ema_decay, int ema_warmup, void* stream) {
  FDBM_REQUIRE(plan && step >= 0 && grad_div > 0.f, "fdbm_plan_optimizer_step: bad arguments");
  if (int rc = plan_guard(plan, "fdbm_plan_optimizer_step")) return rc;
  if (!plan->train) { set_error("fdbm_plan_optimizer_step: not a training plan"); return FDBM_ESTATE; }
  if (plan->ema_swapped) { set_error("fdbm_plan_optimizer_step: the EMA weights are swapped in (restore them first)"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  const int64_t n = plan->params_numel;
  if (int rc = launch_adam_ema(plan->params, plan->grads, plan->adam_m, plan->adam_v, plan->ema, nullptr, n, plan->opt_scratch, grad_div,
                               clip_norm, lr, beta1, beta2, eps, step, ema_decay, ema_warmup, plan->opt_state, s))
    return rc;
  if (int rc = run_pack_ops(plan, s)) return rc;
  return FDBM_OK;
}

extern "C" int fdbm_plan_reset_optimizer(fdbm_plan* plan, void* stream) {
  if (int rc = plan_guard(plan, "fdbm_plan_reset_optimizer")) return rc;
  if (!plan->train) { set_error("fdbm_plan_reset_optimizer: not a training plan"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  const size_t bytes = plan->params_numel * sizeof(float);
  FDBM_CUDA(cudaMemsetAsync(plan->adam_m, 0, bytes, s));
  FDBM_CUDA(cudaMemsetAsync(plan->adam_v, 0, bytes, s));
  FDBM_CUDA(cudaMemcpyAsync(plan->ema, plan->params, bytes, cudaMemcpyDeviceToDevice, s));
  FDBM_CUDA(cudaMemsetAsync(plan->opt_state, 0, 4 * sizeof(double), s));
  plan->ema_swapped = false;
  return FDBM_OK;
}

extern "C" int fdbm_plan_optimizer_state(fdbm_plan* plan, double* out, void* stream) {
  FDBM_REQUIRE(out, "fdbm_plan_optimizer_state: null output");
  if (int rc = plan_guard(plan, "fdbm_plan_optimizer_state")) return rc;
  if (!plan->train) { set_error("fdbm_plan_optimizer_state: not a training plan"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  FDBM_CUDA(cudaMemcpyAsync(out, plan->opt_state, 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  FDBM_CUDA(cudaStreamSynchronize(s));
  return FDBM_OK;
}

extern "C" int fdbm_plan_set_optimizer_state(fdbm_plan* plan, double applied, double skipped, void* stream) {
  if (int rc = plan_guard(plan, "fdbm_plan_set_optimizer_state")) return rc;
  if (!plan->train) { set_error("fdbm_plan_set_optimizer_state: not a training plan"); return FDBM_ESTATE; }
  const double h[4] = {applied, skipped, 0.0, 0.0};
  cudaStream_t s = as_stream(stream);
  FDBM_CUDA(cudaMemcpyAsync(plan->opt_state, h, sizeof(h), cudaMemcpyHostToDevice, s));
  FDBM_CUDA(cudaStreamSynchronize(s));                   // `h` is a stack array
  return FDBM_OK;
}

extern "C" int fdbm_plan_swap_ema(fdbm_plan* plan, int to_ema, void* stream) {
  if (int rc = plan_guard(plan, "fdbm_plan_swap_ema")) return rc;
  if (!plan->train) { set_error("fdbm_plan_swap_ema: not a training plan"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  const size_t bytes = plan->params_numel * sizeof(float);
  if (to_ema) {
    if (plan->ema_swapped) { set_error("fdbm_plan_swap_ema: the EMA weights are already swapped in"); return FDBM_ESTATE; }
    FDBM_CUDA(cudaMemcpyAsync(plan->ema_backup, plan->params, bytes, cudaMemcpyDeviceToDevice, s));
    FDBM_CUDA(cudaMemcpyAsync(plan->params, plan->ema, bytes, cudaMemcpyDeviceToDevice, s));
    plan->ema_swapped = true;
  } else {
    if (!plan->ema_swapped) { set_error("fdbm_plan_swap_ema: nothing to restore"); return FDBM_ESTATE; }
    FDBM_CUDA(cudaMemcpyAsync(plan->params, plan->ema_backup, bytes, cudaMemcpyDeviceToDevice, s));
    plan->ema_swapped = false;
  }
  if (int rc = run_pack_ops(plan, s)) return rc;
  return FDBM_OK;
}

extern "C" int fdbm_plan_destroy(fdbm_plan* plan) {
  if (!plan) return FDBM_OK;
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != plan->device) cudaSetDevice(plan->device);          // frees and destroys must run on the owning device
  if (plan->graph_exec) cudaGraphExecDestroy(plan->graph_exec);
  if (plan->capture_stream) cudaStreamDestroy(plan->capture_stream);
  for (auto& ev : plan->smp_ev) if (ev) cudaEventDestroy(ev);
  cudaFree(plan->smp_y); cudaFree(plan->smp_x); cudaFree(plan->smp_times); cudaFree(plan->smp_coef); cudaFree(plan->smp_rng);
  if (plan->smp_pinned) cudaFreeHost(plan->smp_pinned);
  cudaFree(plan->arena); cudaFree(plan->params); cudaFree(plan->wpacked); cudaFree(plan->d_buf);
  cudaFree(plan->grads); cudaFree(plan->wpacked_d); cudaFree(plan->wgrad_ws);
  cudaFree(plan->adam_m); cudaFree(plan->adam_v); cudaFree(plan->ema); cudaFree(plan->opt_scratch);
  cudaFree(plan->opt_state); cudaFree(plan->ema_backup); cudaFree(plan->pack_descs_d); cudaFree(plan->defer_descs_d); cudaFree(plan->defer_pool);
  if (prev >= 0 && prev != plan->device) cudaSetDevice(prev);
  delete plan;
  return FDBM_OK;
}

extern "C" int fdbm_plan_load_weights(fdbm_plan* plan, const fdbm_tensor_ref* tensors, int n_tensors, void* stream) {
  FDBM_REQUIRE(plan && tensors && n_tensors > 0, "fdbm_plan_load_weights: bad arguments");
  if (int rc = plan_guard(plan, "fdbm_plan_load_weights")) return rc;
  cudaStream_t s = as_stream(stream);
  for (int i = 0; i < n_tensors; ++i) {
    FDBM_REQUIRE(tensors[i].name && tensors[i].data, "fdbm_plan_load_weights: tensor %d has a null field", i);
    auto it = plan->slots.find(tensors[i].name);
    FDBM_REQUIRE(it != plan->slots.end(), "fdbm_plan_load_weights: unexpected tensor '%s'", tensors[i].name);
    FDBM_REQUIRE(it->second.numel == tensors[i].numel, "fdbm_plan_load_weights: '%s' has %lld elements, expected %lld",
                 tensors[i].name, (long long)tensors[i].numel, (long long)it->second.numel);
    FDBM_CUDA(cudaMemcpyAsync(plan->params + it->second.off, tensors[i].data, sizeof(float) * tensors[i].numel,
                              cudaMemcpyDeviceToDevice, s));
    it->second.loaded = true;
  }
  for (auto& kv : plan->slots)
    FDBM_REQUIRE(kv.second.loaded, "fdbm_plan_load_weights: tensor '%s' was never provided", kv.first.c_str());
  if (int rc = run_pack_ops(plan, s)) return rc;
  plan->weights_ready = true;
  return FDBM_OK;
}

extern "C" int64_t fdbm_plan_device_bytes(const fdbm_plan* plan) {
  if (!plan) return 0;
  return plan->arena_bytes + plan->params_numel * 4 + plan->wpacked_bytes + plan->extra_bytes;
}

extern "C" int fdbm_plan_num_launches(const fdbm_plan* plan) { return plan ? plan->n_launches : 0; }

extern "C" int fdbm_ncsnpp_forward(fdbm_plan* plan, const float* x, const float* y, const float* t, float* out,
                                   void* stream) {
  FDBM_REQUIRE(plan && x && out, "fdbm_ncsnpp_forward: null pointer");
  if (int rc = plan_guard(plan, "fdbm_ncsnpp_forward")) return rc;
  if (!plan->weights_ready) { set_error("fdbm_ncsnpp_forward: weights not loaded"); return FDBM_ESTATE; }
  FDBM_REQUIRE(plan->arch.predictive || (y && t), "fdbm_ncsnpp_forward: y and t are required");
  plan->cur_x = x; plan->cur_y = y; plan->cur_t = t; plan->cur_t_stride = 1; plan->cur_out = out;
  return run_ops(plan, as_stream(stream));
}

extern "C" int fdbm_plan_profile_forward(fdbm_plan* plan, const float* x, const float* y, const float* t, float* out,
                                         float* ms, int* kinds, double* flops, int max_ops, void* stream) {
  FDBM_REQUIRE(plan && x && out && ms && kinds && flops, "fdbm_plan_profile_forward: null pointer");
  if (int rc = plan_guard(plan, "fdbm_plan_profile_forward")) return rc;
  if (!plan->weights_ready) { set_error("fdbm_plan_profile_forward: weights not loaded"); return FDBM_ESTATE; }
  FDBM_REQUIRE(plan->arch.predictive || (y && t), "fdbm_plan_profile_forward: y and t are required");
  const int n = static_cast<int>(plan->ops.size());
  FDBM_REQUIRE(max_ops >= n, "fdbm_plan_profile_forward: need room for %d entries", n);
  cudaStream_t s = as_stream(stream);
  plan->cur_x = x; plan->cur_y = y; plan->cur_t = t; plan->cur_t_stride = 1; plan->cur_out = out;
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) FDBM_CUDA(cudaEventCreate(&e));
  int rc = FDBM_OK;
  FDBM_CUDA(cudaEventRecord(ev[0], s));
  for (int i = 0; i < n && rc == FDBM_OK; ++i) {
    rc = plan->ops[i](s);
    if (rc == FDBM_OK && cudaEventRecord(ev[i + 1], s) != cudaSuccess) rc = FDBM_ECUDA;
  }
  if (rc == FDBM_OK && cudaStreamSynchronize(s) != cudaSuccess) rc = cuda_fail(cudaGetLastError(), "cudaStreamSynchronize", __FILE__, __LINE__);
  for (int i = 0; i < n && rc == FDBM_OK; ++i) {
    cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    kinds[i] = plan->op_kind[i];
    flops[i] = plan->op_flops[i];
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc == FDBM_OK ? n : rc;
}

namespace fdbm { int launch_bridge_step_rng(float* x, const float* d, const float* third, const float* coef, int kind,
                                            const uint64_t* rng, uint64_t offset, int64_t n_complex, cudaStream_t s); }

// The N-step loop (fdbm/bridge.py:66-113).  All device memory it needs was allocated by fdbm_plan_create (staging copies
// of y and x, the per-step time / coefficient tables, the Philox seed) and the per-call host arguments travel through a
// plan-owned ring of pinned slots, so this call never allocates and never synchronises in the steady state (it waits on
// a slot's event only if the caller is kRing un-finished calls ahead).  The captured graph reads nothing but plan-owned
// buffers and, for SDE runs with caller-provided noise, the caller's `noise` tensor: a different `noise` address
// re-captures the graph.  A plan serves one host thread at a time.
extern "C" int fdbm_sampler_run(fdbm_plan* plan, const float* y, float* x, const float* times, const float* coef,
                                int n_steps, int kind, const float* noise, uint64_t seed, void* stream) {
  FDBM_REQUIRE(plan && y && x && times && coef && n_steps > 0, "fdbm_sampler_run: bad arguments");
  if (int rc = plan_guard(plan, "fdbm_sampler_run")) return rc;
  FDBM_REQUIRE(!plan->arch.predictive && !plan->train, "fdbm_sampler_run: needs a bridge inference plan (fdbm_plan_create, predictive = 0)");
  FDBM_REQUIRE(kind == FDBM_STEP_ODE || kind == FDBM_STEP_SDE, "fdbm_sampler_run: bad kind");
  FDBM_REQUIRE(n_steps <= fdbm_plan::kMaxSteps, "fdbm_sampler_run: at most %d steps (got %d)", fdbm_plan::kMaxSteps, n_steps);
  if (!plan->weights_ready) { set_error("fdbm_sampler_run: weights not loaded"); return FDBM_ESTATE; }
  cudaStream_t s = as_stream(stream);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  FDBM_CUDA(cudaStreamIsCapturing(s, &cap));
  if (cap != cudaStreamCaptureStatusNone) {
    set_error("fdbm_sampler_run: `stream` is being captured; the sampler owns its CUDA graph and stages host arguments, call it outside a capture");
    return FDBM_ESTATE;
  }
  const int64_t n_complex = static_cast<int64_t>(plan->B) * plan->F_io * plan->T;
  const size_t spec_bytes = static_cast<size_t>(n_complex) * 8;
  const bool want_noise = kind == FDBM_STEP_SDE && noise != nullptr;

  // host arguments -> next pinned slot -> device tables (stream-ordered; the slot is reused kRing calls later)
  const int slot = plan->smp_pos;
  plan->smp_pos = (slot + 1) % fdbm_plan::kRing;
  FDBM_CUDA(cudaEventSynchronize(plan->smp_ev[slot]));
  uint8_t* hs = plan->smp_pinned + kSlotBytes * slot;
  uint64_t* h_rng = reinterpret_cast<uint64_t*>(hs);
  float* h_times = reinterpret_cast<float*>(hs + 16);
  float* h_coef = h_times + fdbm_plan::kMaxSteps;
  h_rng[0] = seed; h_rng[1] = 0;
  FDBM_CUDA(cudaMemcpyAsync(plan->smp_rng, h_rng, 16, cudaMemcpyHostToDevice, s));
  const std::vector<float> ht(times, times + n_steps), hc(coef, coef + 3 * n_steps);
  if (ht != plan->smp_h_times || hc != plan->smp_h_coef) {
    std::copy(ht.begin(), ht.end(), h_times);
    std::copy(hc.begin(), hc.end(), h_coef);
    FDBM_CUDA(cudaMemcpyAsync(plan->smp_times, h_times, sizeof(float) * n_steps, cudaMemcpyHostToDevice, s));
    FDBM_CUDA(cudaMemcpyAsync(plan->smp_coef, h_coef, sizeof(float) * 3 * n_steps, cudaMemcpyHostToDevice, s));
    plan->smp_h_times = ht; plan->smp_h_coef = hc;
  }
  FDBM_CUDA(cudaEventRecord(plan->smp_ev[slot], s));
  FDBM_CUDA(cudaMemcpyAsync(plan->smp_y, y, spec_bytes, cudaMemcpyDeviceToDevice, s));
  FDBM_CUDA(cudaMemcpyAsync(plan->smp_x, x, spec_bytes, cudaMemcpyDeviceToDevice, s));

  GraphKey key{{plan->smp_y, plan->smp_x, plan->smp_times, plan->smp_coef, want_noise ? noise : nullptr, nullptr}, n_steps, kind, 0};
  if (!(plan->have_graph && plan->graph_key == key)) {
    if (plan->graph_exec) { cudaGraphExecDestroy(plan->graph_exec); plan->graph_exec = nullptr; plan->have_graph = false; }
    cudaGraph_t graph = nullptr;
    cudaStream_t cs = plan->capture_stream;
    FDBM_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    int rc = FDBM_OK;
    for (int i = 0; i < n_steps && rc == FDBM_OK; ++i) {
      plan->cur_x = plan->smp_x; plan->cur_y = plan->smp_y; plan->cur_t = plan->smp_times + i; plan->cur_t_stride = 0; plan->cur_out = plan->d_buf;
      rc = run_ops(plan, cs);
      const float* third = kind == FDBM_STEP_ODE ? plan->smp_y : (want_noise ? noise + 2 * n_complex * i : nullptr);
      if (rc == FDBM_OK)
        rc = launch_bridge_step_rng(plan->smp_x, plan->d_buf, third, plan->smp_coef + 3 * i, kind, plan->smp_rng,
                                    static_cast<uint64_t>(i) + 1, n_complex, cs);
    }
    const cudaError_t e = cudaStreamEndCapture(cs, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) return cuda_fail(e, "cudaStreamEndCapture", __FILE__, __LINE__);
    const cudaError_t e2 = cudaGraphInstantiate(&plan->graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e2 != cudaSuccess) return cuda_fail(e2, "cudaGraphInstantiate", __FILE__, __LINE__);
    plan->graph_key = key; plan->have_graph = true;
  }
  FDBM_CUDA(cudaGraphLaunch(plan->graph_exec, s));
  FDBM_CUDA(cudaMemcpyAsync(x, plan->smp_x, spec_bytes, cudaMemcpyDeviceToDevice, s));
  return FDBM_OK;
}
