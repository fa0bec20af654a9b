// mmd_bifpn_run: resolve an op list (include/mmd.h) into kernel arguments and enqueue it on the caller's stream.
#include <vector>

#include "bifpn.cuh"

namespace mmd {

static TensorP resolve(const MmdTensor& t, const Bases& B) {
  TensorP r;
  r.data = B.get<void>(t.data);
  r.bn = B.get<float>(t.bn);
  r.H = t.H;
  r.W = t.W;
  return r;
}

static int fill_fwd(const MmdOp& op, const Bases& B, int batch, NodeFwdP& p) {
  MMD_CHECK_ARG(op.n_in >= 1 && op.n_in <= 3, "op: n_in=%d", op.n_in);
  for (int i = 0; i < 3; ++i) {
    p.in[i] = (i < op.n_in) ? resolve(op.in[i], B) : TensorP{nullptr, nullptr, 0, 0};
    p.mode[i] = op.mode[i];
    p.pidx[i] = B.get<unsigned char>(op.pidx[i]);
    if (i < op.n_in) MMD_CHECK_ARG(p.in[i].data != nullptr, "op: input %d has no data", i);
  }
  p.n_in = op.n_in;
  p.swish = op.swish;
  p.train = op.train;
  p.Cin = op.Cin;
  p.fw = op.fw;
  p.fw_eps = op.fw_eps;
  p.fw_n = op.fw_n;
  for (int i = 0; i < 3; ++i) p.fw_idx[i] = op.fw_idx[i];
  p.dw_w = op.dw_w; p.pw_w = op.pw_w; p.pw_b = op.pw_b; p.bn_w = op.bn_w; p.bn_b = op.bn_b;
  p.bn_rm = op.bn_rm; p.bn_rv = op.bn_rv; p.bn_nbt = (long long*)op.bn_nbt;
  p.out = B.get<void>(op.out.data);
  p.out_bn = B.get<float>(op.out.bn);
  p.save_d = B.get<void>(op.save_d);
  p.packed = B.get<unsigned char>(op.packed);
  p.stats = B.get<double>(op.stats);
  p.counter = B.get<unsigned>(op.counter);
  p.bn_eps = op.bn_eps;
  p.bn_mom = op.bn_momentum;
  p.g = make_geom(batch, op.out.H, op.out.W);
  p.defer_bn = 0;
  p.frozen_bn = 0;
  for (int i = 0; i < 3; ++i) p.bnsrc[i] = BnSrc{nullptr, nullptr, nullptr, 0.0, 0.f};
  MMD_CHECK_ARG(p.out != nullptr, "op: no output");
  if (op.kind != MMD_OP_BNAPPLY && op.kind != MMD_OP_POOLFUSE) {
    MMD_CHECK_ARG(p.pw_w && p.pw_b && p.bn_w && p.bn_b && p.bn_rm && p.bn_rv, "op: missing conv/bn parameters");
    if (op.train) MMD_CHECK_ARG(p.out_bn && p.stats && p.counter, "train op: missing bn/stats/counter storage");
    MMD_CHECK_ARG(!op.frozen_bn || (op.train && p.out_bn), "op: a frozen BatchNorm needs train = 1 and a BatchNorm vector");
    p.frozen_bn = op.frozen_bn ? 1 : 0;
  }
  return 0;
}

static int fill_bwd(const MmdOp& op, const Bases& B, int batch, NodeBwdP& p) {
  for (int i = 0; i < 3; ++i) {
    p.in[i] = (i < op.n_in) ? resolve(op.in[i], B) : TensorP{nullptr, nullptr, 0, 0};
    p.mode[i] = op.mode[i];
    p.in_bn_w[i] = op.in_bn_w[i];
    p.in_bn_b[i] = op.in_bn_b[i];
    p.pidx[i] = B.get<unsigned char>(op.pidx[i]);
    p.in_slot[i] = B.get<double>(op.in_slot[i]);
  }
  p.n_in = op.n_in;
  p.swish = op.swish;
  p.Cin = op.Cin;
  p.accumulate_dx = op.accumulate_dx;
  p.fw = op.fw;
  p.fw_eps = op.fw_eps;
  p.dw_w = op.dw_w; p.pw_w = op.pw_w; p.bn_w = op.bn_w;
  p.out = B.get<void>(op.out.data);
  p.out_bn = B.get<float>(op.out.bn);
  p.save_d = B.get<void>(op.save_d);
  p.packed = B.get<unsigned char>(op.packed);
  p.aux = B.get<void>(op.aux);
  p.praw = B.get<void>(op.praw);
  p.n_cons = op.n_cons;
  MMD_CHECK_ARG(op.n_cons >= 0 && op.n_cons <= 3, "op: n_cons=%d", op.n_cons);
  for (int c = 0; c < 3; ++c) {
    ConsP& cs = p.cons[c];
    if (c < op.n_cons) {
      const MmdCons& m = op.cons[c];
      cs.du = B.get<void>(m.du.data);
      cs.H = m.du.H; cs.W = m.du.W;
      cs.mode = m.mode;
      cs.fw_k = m.fw_k; cs.fw_n = m.fw_n; cs.fw_eps = m.fw_eps; cs.fw = m.fw;
      cs.slot = B.get<double>(m.slot);
      cs.pidx = B.get<unsigned char>(m.pidx);
      MMD_CHECK_ARG(cs.du != nullptr, "op: consumer %d has no gradient tensor", c);
      if (cs.mode == MMD_CONS_POOL) MMD_CHECK_ARG(cs.pidx != nullptr, "op: pooled consumer %d has no arg-max indices", c);
    } else {
      cs = ConsP{nullptr, 0, 0, 0, 0, 0, 0.f, nullptr, nullptr, nullptr};
    }
  }
  p.du = B.get<void>(op.du);
  p.dd = B.get<void>(op.dd);
  p.dx = B.get<void>(op.dx);
  p.g_dw = B.get<float>(op.g_dw); p.g_pw = B.get<float>(op.g_pw); p.g_pb = B.get<float>(op.g_pb);
  p.g_bn_w = B.get<float>(op.g_bn_w); p.g_bn_b = B.get<float>(op.g_bn_b); p.g_fw = B.get<float>(op.g_fw);
  p.counter = B.get<unsigned>(op.counter);
  p.g = make_geom(batch, op.out.H, op.out.W);
  p.defer_fw = 0;
  p.frozen_bn = (op.kind == MMD_OP_NODE_BWD || op.kind == MMD_OP_PROJ_BWD) && op.frozen_bn ? 1 : 0;
  return 0;
}

// ---- deferred BatchNorm finalisation plan of one forward op list (see NodeFwdP::defer_bn) ------------------------------
struct DeferPlan {
  std::vector<char> defer;                 // per op: the producer skips its in-kernel finalisation
  std::vector<BnSrc> src;                  // per op and input (3 per op): where a consumer rebuilds (scale, shift) from
  std::vector<BnFinalEntry> fin;           // what bn_finalize_all has to do at the end of the list
  bool any() const { return !fin.empty(); }
};

static bool ref_eq(const MmdRef& a, const MmdRef& b) { return a.base >= 0 && a.base == b.base && a.off == b.off; }

// A train-mode NODE_FWD / PROJ_FWD op may defer when every later op that applies its BatchNorm on load runs on a kernel
// that can rebuild the coefficients from the statistics: the v4 node kernel, the poolfuse pre-pass, bnapply.  A frozen
// BatchNorm has no statistics: its vector is written before the forward and its consumers read it as it is.
static int plan_defer(const MmdOp* ops, int n_ops, const Bases& B, int batch, int dtype, DeferPlan& D) {
  D.defer.assign(n_ops, 0);
  D.src.assign((size_t)n_ops * 3, BnSrc{nullptr, nullptr, nullptr, 0.0, 0.f});
  D.fin.clear();
  if (dtype != MMD_BF16 || tc_disabled() || !bn_deferral_enabled()) return 0;
  for (int j = 0; j < n_ops; ++j) {
    const MmdOp& op = ops[j];
    if (!op.train || op.frozen_bn || !(op.kind == MMD_OP_NODE_FWD || (op.kind == MMD_OP_PROJ_FWD && op.Cin % 8 == 0))) continue;
    if (op.out.bn.base < 0 || op.stats.base < 0) continue;
    bool ok = true;
    for (int k = j + 1; k < n_ops && ok; ++k) {
      const MmdOp& ck = ops[k];
      bool reads = false;
      for (int i = 0; i < ck.n_in && i < 3; ++i) reads = reads || ref_eq(ck.in[i].bn, op.out.bn);
      if (!reads) continue;
      if (ck.kind == MMD_OP_POOLFUSE || ck.kind == MMD_OP_BNAPPLY) continue;
      if (ck.kind != MMD_OP_NODE_FWD) { ok = false; break; }
      NodeFwdP cp;
      int rc = fill_fwd(ck, B, batch, cp);
      if (rc) return rc;
      if (!fwd_v4_usable(cp)) ok = false;
    }
    if (!ok) continue;
    BnFinalEntry e;
    e.stats = B.get<double>(op.stats);
    e.gamma = op.bn_w; e.beta = op.bn_b;
    e.rm = op.bn_rm; e.rv = op.bn_rv; e.nbt = (long long*)op.bn_nbt;
    e.out_bn = B.get<float>(op.out.bn);
    e.n = (double)batch * op.out.H * op.out.W;
    e.eps = op.bn_eps; e.mom = op.bn_momentum;
    if (e.stats == nullptr || e.out_bn == nullptr || e.gamma == nullptr || e.beta == nullptr || e.rm == nullptr || e.rv == nullptr) continue;
    D.defer[j] = 1;
    D.fin.push_back(e);
    for (int k = j + 1; k < n_ops; ++k)
      for (int i = 0; i < ops[k].n_in && i < 3; ++i)
        if (ref_eq(ops[k].in[i].bn, op.out.bn)) D.src[(size_t)k * 3 + i] = BnSrc{e.stats, e.gamma, e.beta, e.n, e.eps};
  }
  return 0;
}

static void apply_defer(const DeferPlan* D, int idx, NodeFwdP& p) {
  if (D == nullptr || D->defer.empty()) return;
  p.defer_bn = D->defer[idx];
  for (int i = 0; i < 3; ++i) p.bnsrc[i] = D->src[(size_t)idx * 3 + i];
}

// entries of the deferred fusion-weight gradient launch collected while an op list runs (see FwGradEntry)
struct FwGradList {
  FwGradEntry e[128];
  int n = 0;
};

}  // namespace mmd

using namespace mmd;

static int run_one(const MmdOp& op, int i, const Bases& B, int batch, int C, int dtype, cudaStream_t stream,
                   FwGradList* fwl = nullptr, const DeferPlan* dp = nullptr);

static bool same_ref(const MmdRef& a, const MmdRef& b) { return a.base >= 0 && a.base == b.base && a.off == b.off; }

// Number of consecutive ops starting at `i` that may share ONE launch: BNAPPLY ops none of which reads the output of an
// earlier one of the run (the 5 output normalisations of a training stack), or SLOT ops (always independent).
static int group_len(const MmdOp* ops, int i, int n_ops) {
  const int kind = ops[i].kind;
  if (kind != MMD_OP_BNAPPLY && kind != MMD_OP_SLOT) return 1;
  int n = 1;
  while (i + n < n_ops && n < kMaxGroupOps && ops[i + n].kind == kind) {
    bool dep = false;
    if (kind == MMD_OP_BNAPPLY)
      for (int k = 0; k < n; ++k) dep = dep || same_ref(ops[i + n].in[0].data, ops[i + k].out.data);
    if (dep) break;
    ++n;
  }
  return n;
}

// launches ops[i .. i+n) (n >= 2, from group_len) together
static int run_group(const MmdOp* ops, int i, int n, const Bases& B, int batch, int C, int dtype, cudaStream_t stream,
                     const DeferPlan* dp = nullptr) {
  int rc = 0;
  if (ops[i].kind == MMD_OP_BNAPPLY) {
    NodeFwdP ps[kMaxGroupOps];
    for (int k = 0; k < n; ++k) {
      if ((rc = fill_fwd(ops[i + k], B, batch, ps[k]))) return rc;
      apply_defer(dp, i + k, ps[k]);
    }
    return launch_bnapply_group(ps, n, C, dtype, stream);
  }
  NodeBwdP ps[kMaxGroupOps];
  for (int k = 0; k < n; ++k) {
    const MmdOp& op = ops[i + k];
    if ((rc = fill_bwd(op, B, batch, ps[k]))) return rc;
    MMD_CHECK_ARG(ps[k].in[0].data && ps[k].in[0].bn && ps[k].in_slot[0] && op.n_cons == 1, "slot op %d: missing storage", i + k);
    if (op.mode[0] == MMD_IN_POOL) MMD_CHECK_ARG(ps[k].pidx[0] != nullptr, "slot op %d: no arg-max indices", i + k);
  }
  return launch_slot_group(ps, n, C, dtype, stream);
}

// ---- persistent small-level chains (bifpn.cuh: ChainStepH) -------------------------------------------------------------
// Starting at op index i of every member list (lists whose ops line up), collect consecutive units — NODE_FWD, or POOLFUSE
// followed by the NODE_FWD that consumes it — that the chain kernel can run (P5 and smaller, v4 bodies, deferred BatchNorm
// when training) and launch them as ONE kernel.  Returns the number of op-list entries consumed (0: no chain, nothing
// launched); *rc carries a launch error.
static int try_chain_fwd(const MmdOp* const* ops, const int32_t* n_ops, void* const* const* bases, const int32_t* n_bases,
                         const DeferPlan* plans, const int* members, int n_members, int i, int batch, int C, int dtype,
                         cudaStream_t stream, int* rc) {
  *rc = 0;
  if (dtype != MMD_BF16 || tc_disabled() || !chain_fwd_enabled() || n_members < 1) return 0;
  static thread_local ChainStepH steps[kMaxChainStepsH];
  int n_steps = 0, j = i;
  const int m0 = members[0];
  while (n_steps < kMaxChainStepsH && j < n_ops[m0]) {
    const MmdOp& a = ops[m0][j];
    int len, node_at;
    if (a.kind == MMD_OP_POOLFUSE && j + 1 < n_ops[m0] && ops[m0][j + 1].kind == MMD_OP_NODE_FWD) { len = 2; node_at = j + 1; }
    else if (a.kind == MMD_OP_NODE_FWD) { len = 1; node_at = j; }
    else break;
    if (ops[m0][node_at].out.H * ops[m0][node_at].out.W > 24 * 24) break;
    static const int max_pre_hw = (int)env_float("MMD_CHAIN_PRE_MAX_HW", 24.f * 24.f);   // largest level pooled inline
    if (len == 2 && ops[m0][node_at].out.H * ops[m0][node_at].out.W > max_pre_hw) break;
    ChainStepH& st = steps[n_steps];
    st.has_pre = (len == 2) ? 1 : 0;
    bool ok = true;
    for (int k = 0; k < n_members && ok; ++k) {
      const int m = members[k];
      if (j + len > n_ops[m]) { ok = false; break; }
      const MmdOp& om = ops[m][node_at];
      if (om.kind != MMD_OP_NODE_FWD || om.out.H != ops[m0][node_at].out.H || om.out.W != ops[m0][node_at].out.W) { ok = false; break; }
      if (len == 2 && ops[m][j].kind != MMD_OP_POOLFUSE) { ok = false; break; }
      if (len == 1 && ops[m][j].kind != MMD_OP_NODE_FWD) { ok = false; break; }
      Bases Bm{bases[m], n_bases[m]};
      if (fill_fwd(om, Bm, batch, st.node[k]) != 0) { ok = false; break; }
      apply_defer(&plans[m], node_at, st.node[k]);
      if (len == 2) {
        if (fill_fwd(ops[m][j], Bm, batch, st.pre[k]) != 0) { ok = false; break; }
        apply_defer(&plans[m], j, st.pre[k]);
      } else {
        st.pre[k] = st.node[k];
      }
      if (!chain_fwd_step_usable(st.node[k], len == 2 ? &st.pre[k] : nullptr)) ok = false;
    }
    if (!ok) break;
    if (n_steps == 0 && steps[0].node[0].counter == nullptr) break;   // the barrier words live in the first node's counter
    ++n_steps;
    j += len;
  }
  if (n_steps < 2) return 0;
  *rc = launch_chain_fwd(steps, n_steps, n_members, C, stream);
  return j - i;
}

extern "C" int mmd_bifpn_run_multi(const MmdOp* const* ops, const int32_t* n_ops, void* const* const* bases,
                                   const int32_t* n_bases, int32_t n_lists, int32_t batch, int32_t C, int32_t dtype,
                                   mmd_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMD_CHECK_ARG(ops && n_ops && bases && n_bases && n_lists >= 1 && n_lists <= kMaxBatchNets, "mmd_bifpn_run_multi: bad arguments");
  MMD_CHECK_ARG(batch >= 1 && C == 112, "mmd_bifpn_run_multi: batch=%d C=%d", batch, C);
  MMD_CHECK_ARG(dtype == MMD_F32 || dtype == MMD_BF16, "mmd_bifpn_run_multi: dtype %d", dtype);
  int max_n = 0;
  for (int l = 0; l < n_lists; ++l) max_n = n_ops[l] > max_n ? n_ops[l] : max_n;
  int grouped_until[kMaxBatchNets] = {0, 0, 0, 0};   // ops below this index already ran as part of a group launch
  DeferPlan plans[kMaxBatchNets];
  for (int l = 0; l < n_lists; ++l) {
    Bases Bl{bases[l], n_bases[l]};
    int rc = plan_defer(ops[l], n_ops[l], Bl, batch, dtype, plans[l]);
    if (rc) return rc;
  }
  for (int i = 0; i < max_n; ++i) {
    bool done[kMaxBatchNets] = {false, false, false, false};
    for (int l = 0; l < n_lists; ++l) {
      if (done[l] || i >= n_ops[l] || i < grouped_until[l]) continue;
      const MmdOp& op = ops[l][i];
      const bool batchable = (dtype == MMD_BF16 && !tc_disabled() &&
                              (op.kind == MMD_OP_NODE_FWD || op.kind == MMD_OP_POOLFUSE ||
                               (op.kind == MMD_OP_PROJ_FWD && op.Cin % 8 == 0))) ||
                             op.kind == MMD_OP_BNAPPLY;
      NodeFwdP ps[kMaxBatchNets];
      int members[kMaxBatchNets], n = 0;
      // a run of small-level nodes of all lockstep networks: ONE persistent launch (try_chain_fwd)
      if (op.kind == MMD_OP_NODE_FWD || op.kind == MMD_OP_POOLFUSE) {
        for (int m = l; m < n_lists; ++m) {
          if (done[m] || i >= n_ops[m] || i < grouped_until[m]) continue;
          const MmdOp& om = ops[m][i];
          if (om.kind != op.kind || om.out.H != op.out.H || om.out.W != op.out.W) continue;
          members[n++] = m;
        }
        int rc = 0;
        const int used = try_chain_fwd(ops, n_ops, bases, n_bases, plans, members, n, i, batch, C, dtype, stream, &rc);
        if (rc) return rc;
        if (used > 0) {
          for (int k = 0; k < n; ++k) {
            done[members[k]] = true;
            grouped_until[members[k]] = i + used;
          }
          continue;
        }
        n = 0;
      }
      // POOLFUSE followed by the node that consumes it, small level: ONE launch (the node kernel pools inline)
      if (dtype == MMD_BF16 && !tc_disabled() && op.kind == MMD_OP_POOLFUSE && i + 1 < n_ops[l] &&
          ops[l][i + 1].kind == MMD_OP_NODE_FWD) {
        NodeFwdP nodes[kMaxBatchNets];
        for (int m = l; m < n_lists; ++m) {
          if (done[m] || i + 1 >= n_ops[m] || i < grouped_until[m]) continue;
          const MmdOp& om = ops[m][i];
          const MmdOp& on = ops[m][i + 1];
          if (om.kind != MMD_OP_POOLFUSE || on.kind != MMD_OP_NODE_FWD || om.out.H != op.out.H || om.out.W != op.out.W) continue;
          Bases Bm{bases[m], n_bases[m]};
          int rc = fill_fwd(om, Bm, batch, ps[n]);
          if (rc) return rc;
          if ((rc = fill_fwd(on, Bm, batch, nodes[n]))) return rc;
          apply_defer(&plans[m], i, ps[n]);
          apply_defer(&plans[m], i + 1, nodes[n]);
          if (!fwd_v4_pre_usable(ps[n], nodes[n])) continue;
          members[n++] = m;
        }
        if (n >= 1 && members[0] == l) {
          int rc = launch_node_fwd_v4_pre(nodes, ps, n, C, stream);
          if (rc) return rc;
          for (int k = 0; k < n; ++k) {
            done[members[k]] = true;
            grouped_until[members[k]] = i + 2;
          }
          continue;
        }
        n = 0;
      }
      if (batchable) {
        for (int m = l; m < n_lists; ++m) {
          if (done[m] || i >= n_ops[m] || i < grouped_until[m]) continue;
          const MmdOp& om = ops[m][i];
          if (om.kind != op.kind || om.out.H != op.out.H || om.out.W != op.out.W || om.Cin != op.Cin) continue;
          if (op.kind == MMD_OP_BNAPPLY && (om.mode[0] != op.mode[0] || om.in[0].H != op.in[0].H || om.in[0].W != op.in[0].W)) continue;
          Bases Bm{bases[m], n_bases[m]};
          int rc = fill_fwd(om, Bm, batch, ps[n]);
          if (rc) return rc;
          apply_defer(&plans[m], i, ps[n]);
          if (op.kind == MMD_OP_NODE_FWD && !fwd_v4_usable(ps[n])) continue;
          members[n++] = m;
        }
      }
      if (n >= 2) {
        int rc = (op.kind == MMD_OP_NODE_FWD)   ? launch_node_fwd_v4(ps, n, C, stream)
                 : (op.kind == MMD_OP_POOLFUSE) ? launch_poolfuse(ps, n, C, stream)
                 : (op.kind == MMD_OP_BNAPPLY)  ? launch_bnapply_multi(ps, n, C, dtype, stream)
                                                : launch_proj_fwd_tc_multi(ps, n, C, stream);
        if (rc) return rc;
        for (int k = 0; k < n; ++k) done[members[k]] = true;
      }
      if (!done[l]) {
        Bases Bl{bases[l], n_bases[l]};
        const int g = group_len(ops[l], i, n_ops[l]);
        int rc = (g >= 2) ? run_group(ops[l], i, g, Bl, batch, C, dtype, stream, &plans[l])
                          : run_one(op, i, Bl, batch, C, dtype, stream, nullptr, &plans[l]);
        if (rc) return rc;
        if (g >= 2) grouped_until[l] = i + g;
        done[l] = true;
      }
    }
  }
  for (int l = 0; l < n_lists; ++l)   // every forward consumer has run: finalise the deferred BatchNorms of each list
    if (plans[l].any()) {
      int rc = launch_bn_finalize_all(plans[l].fin.data(), (int)plans[l].fin.size(), C, stream);
      if (rc) return rc;
    }
  return 0;
}

extern "C" int mmd_bifpn_run(const MmdOp* ops, int32_t n_ops, void* const* bases, int32_t n_bases, int32_t batch,
                             int32_t C, int32_t dtype, mmd_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMD_CHECK_ARG(ops != nullptr && n_ops >= 0 && bases != nullptr, "mmd_bifpn_run: null arguments");
  MMD_CHECK_ARG(batch >= 1, "mmd_bifpn_run: batch=%d", batch);
  MMD_CHECK_ARG(C == 112, "mmd_bifpn_run: kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(dtype == MMD_F32 || dtype == MMD_BF16, "mmd_bifpn_run: dtype %d", dtype);
  Bases B{bases, n_bases};
  FwGradList fwl;
  DeferPlan plan;
  {
    int rc = plan_defer(ops, n_ops, B, batch, dtype, plan);
    if (rc) return rc;
  }
  for (int i = 0; i < n_ops;) {
    if (ops[i].kind == MMD_OP_NODE_FWD || ops[i].kind == MMD_OP_POOLFUSE) {   // a run of small-level nodes: one launch
      const int member = 0;
      const MmdOp* lists[1] = {ops};
      const int32_t counts[1] = {n_ops};
      void* const* blists[1] = {bases};
      const int32_t bcounts[1] = {n_bases};
      int rc = 0;
      const int used = try_chain_fwd(lists, counts, blists, bcounts, &plan, &member, 1, i, batch, C, dtype, stream, &rc);
      if (rc) return rc;
      if (used > 0) {
        i += used;
        continue;
      }
    }
    if (dtype == MMD_BF16 && !tc_disabled() && ops[i].kind == MMD_OP_POOLFUSE && i + 1 < n_ops && ops[i + 1].kind == MMD_OP_NODE_FWD) {
      NodeFwdP pre, node;
      int rc = fill_fwd(ops[i], B, batch, pre);
      if (rc) return rc;
      if ((rc = fill_fwd(ops[i + 1], B, batch, node))) return rc;
      apply_defer(&plan, i, pre);
      apply_defer(&plan, i + 1, node);
      if (fwd_v4_pre_usable(pre, node)) {
        if ((rc = launch_node_fwd_v4_pre(&node, &pre, 1, C, stream))) return rc;
        i += 2;
        continue;
      }
    }
    const int g = group_len(ops, i, n_ops);
    int rc = (g >= 2) ? run_group(ops, i, g, B, batch, C, dtype, stream, &plan) : run_one(ops[i], i, B, batch, C, dtype, stream, &fwl, &plan);
    if (rc) return rc;
    i += g;
  }
  if (plan.any()) {   // every forward consumer has run: finalise the deferred BatchNorms
    int rc = launch_bn_finalize_all(plan.fin.data(), (int)plan.fin.size(), C, stream);
    if (rc) return rc;
  }
  if (fwl.n > 0) return launch_fwgrad(fwl.e, fwl.n, C, stream);   // all slots are complete: every g_fw in one launch
  return 0;
}

static int run_one(const MmdOp& op, int i, const Bases& B, int batch, int C, int dtype, cudaStream_t stream, FwGradList* fwl,
                   const DeferPlan* dp) {
  int rc = 0;
    switch (op.kind) {
    case MMD_OP_NODE_FWD:
    case MMD_OP_PROJ_FWD:
    case MMD_OP_POOLFUSE:
    case MMD_OP_BNAPPLY: {
      NodeFwdP p;
      if ((rc = fill_fwd(op, B, batch, p))) return rc;
      apply_defer(dp, i, p);
      if (op.kind == MMD_OP_NODE_FWD) {
        MMD_CHECK_ARG(p.dw_w != nullptr, "node op %d: no depthwise weight", i);
        for (int k = 0; k < op.n_in; ++k) MMD_CHECK_ARG(op.in[k].C == C, "node op %d: input %d has C=%d", i, k, op.in[k].C);
        rc = launch_node_fwd(p, C, dtype, stream);
      } else if (op.kind == MMD_OP_PROJ_FWD) {
        MMD_CHECK_ARG(op.Cin >= 4 && op.Cin % 4 == 0, "proj op %d: Cin=%d must be a positive multiple of 4", i, op.Cin);
        rc = launch_proj_fwd(p, C, dtype, stream);
      } else if (op.kind == MMD_OP_POOLFUSE) {
        MMD_CHECK_ARG(dtype == MMD_BF16, "poolfuse op %d: bf16 plans only", i);
        rc = launch_poolfuse(&p, 1, C, stream);
      } else {
        rc = launch_bnapply(p, C, dtype, stream);
      }
      break;
    }
    case MMD_OP_NODE_BWD:
    case MMD_OP_PROJ_BWD:
    case MMD_OP_PULL:
    case MMD_OP_SLOT: {
      NodeBwdP p;
      if ((rc = fill_bwd(op, B, batch, p))) return rc;
      if (op.kind == MMD_OP_NODE_BWD) {
        MMD_CHECK_ARG(p.out && p.out_bn && p.save_d && p.du && p.dd && p.g_pw && p.counter, "node bwd op %d: missing storage", i);
        if (fwl != nullptr && fwl->n < 128 && dtype == MMD_BF16 && !tc_disabled() && fwgrad_deferral_enabled() &&
            p.fw != nullptr && p.g_fw != nullptr && bwd_v4_usable(p)) {
          FwGradEntry& e = fwl->e[fwl->n];
          bool ok = true;
          for (int k = 0; k < 3; ++k) {
            e.slot[k] = (k < p.n_in) ? p.in_slot[k] : nullptr;
            e.in_bn_w[k] = (k < p.n_in && p.in[k].bn != nullptr) ? p.in_bn_w[k] : nullptr;
            e.in_bn_b[k] = (k < p.n_in && p.in[k].bn != nullptr) ? p.in_bn_b[k] : nullptr;
            if (k < p.n_in && p.in_slot[k] == nullptr) ok = false;
            if (k < p.n_in && p.in[k].bn != nullptr && (p.in_bn_w[k] == nullptr || p.in_bn_b[k] == nullptr)) ok = false;
          }
          e.fw = p.fw; e.g_fw = p.g_fw; e.fw_eps = p.fw_eps; e.n_in = p.n_in;
          if (ok) {
            p.defer_fw = 1;
            ++fwl->n;
          }
        }
        rc = launch_node_bwd(p, C, dtype, stream);
      } else if (op.kind == MMD_OP_PROJ_BWD) {
        MMD_CHECK_ARG(p.out && p.out_bn && p.g_pw && p.in[0].data, "proj bwd op %d: missing storage", i);
        rc = launch_proj_bwd(p, C, dtype, stream);
      } else if (op.kind == MMD_OP_PULL) {
        MMD_CHECK_ARG(p.dx != nullptr, "pull op %d: no destination", i);
        rc = launch_pull(p, C, dtype, stream);
      } else {
        MMD_CHECK_ARG(p.in[0].data && p.in[0].bn && p.in_slot[0] && op.n_cons == 1, "slot op %d: missing storage", i);
        if (op.mode[0] == MMD_IN_POOL) MMD_CHECK_ARG(p.pidx[0] != nullptr, "slot op %d: no arg-max indices", i);
        rc = launch_slot(p, C, dtype, stream);
      }
      break;
    }
    case MMD_OP_COPY:   // executed by mmd_bifpn_prep
      break;
    case MMD_OP_ACT_FWD:
    case MMD_OP_ACT_BWD: {
      const long long n = (long long)batch * op.in[0].H * op.in[0].W * C;
      MMD_CHECK_ARG(op.n_in == 1 && op.in[0].C == C && op.in[0].bn.base < 0, "act op %d: one final C-channel input expected", i);
      if (op.kind == MMD_OP_ACT_FWD)
        rc = launch_act_fwd(B.get<void>(op.in[0].data), B.get<void>(op.out.data), n, dtype, stream);
      else
        rc = launch_act_bwd(B.get<void>(op.in[0].data), op.n_cons == 1 ? B.get<void>(op.cons[0].du.data) : nullptr,
                            B.get<void>(op.dx), n, dtype, stream);
      break;
    }
    case MMD_OP_HEAD_GATHER:
    case MMD_OP_HEAD_SCATTER: {
      const bool scatter = op.kind == MMD_OP_HEAD_SCATTER;
      MMD_CHECK_ARG(op.n_in >= 1 && op.n_in <= 2 && op.n_in == (op.head_K + C - 1) / C, "head op %d: n_in=%d for K=%d", i, op.n_in, op.head_K);
      const void* in[2] = {B.get<void>(op.in[0].data), op.n_in > 1 ? B.get<void>(op.in[1].data) : nullptr};
      void* dst[2] = {B.get<void>(op.du), B.get<void>(op.dd)};
      rc = launch_head_move(scatter ? 1 : 0, in, dst, B.get<void>(op.out.data),
                            scatter && op.n_cons == 1 ? B.get<void>(op.cons[0].du.data) : nullptr, batch,
                            op.in[0].H * op.in[0].W, C, op.head_K, op.head_tot, op.head_off, op.head_act, dtype, stream);
      break;
    }
    default:
      set_error("mmd_bifpn_run: op %d has unknown kind %d", i, op.kind);
      return MMD_E_ARG;
  }
  return rc;
}
