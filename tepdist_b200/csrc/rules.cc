#include "rules.h"

#include <algorithm>
#include <functional>
#include <set>

namespace tepdist {
namespace {

using DS = DimStrategy;

struct Ctx {
  const Graph& g;
  const Node& n;
  int num;
  std::vector<Candidate> out;

  const TensorType& in(int i) const { return g.type(n.inputs[i]); }
  const TensorType& o(int i = 0) const { return n.outputs[i]; }
  int nin() const { return (int)n.inputs.size(); }
  bool divisible(const TensorType& t, int d) const { return d >= 0 && d < t.rank() && t.dims[d] % num == 0 && t.dims[d] >= num; }
  DS S(int d) const { return DS::Split(d, num); }
  DS P(int kind = 0) const { return DS::Partial(num, kind); }
  static DS G() { return DS::Glue(); }

  void add(std::vector<DS> ins, std::vector<DS> outs, const std::string& tag, double cost = 0) {
    // validate divisibility of every split
    for (int i = 0; i < (int)ins.size(); ++i)
      if (ins[i].is_split() && !ins[i].Valid(in(i))) return;
    for (int i = 0; i < (int)outs.size(); ++i)
      if (outs[i].is_split() && !outs[i].Valid(o(i))) return;
    Candidate c;
    c.ins = std::move(ins);
    c.outs = std::move(outs);
    c.tag = tag;
    c.node_cost = cost;
    out.push_back(std::move(c));
  }
  void add_glue() {
    add(std::vector<DS>(nin(), G()), std::vector<DS>(n.outputs.size(), G()), "glue");
  }
};

// operand strategy that corresponds to output split on dim d under numpy-style (right-aligned) broadcasting
DS BroadcastOperand(const TensorType& operand, const TensorType& out, int d, int num) {
  int od = d - (out.rank() - operand.rank());
  if (od < 0 || operand.dims[od] != out.dims[d]) return DS::Glue();
  return DS::Split(od, num);
}

void Elementwise(Ctx& c, bool linear_in_all_operands) {
  const TensorType& o = c.o();
  for (int d = 0; d < o.rank(); ++d) {
    if (!c.divisible(o, d)) continue;
    std::vector<DS> ins;
    for (int i = 0; i < c.nin(); ++i) ins.push_back(BroadcastOperand(c.in(i), o, d, c.num));
    c.add(ins, std::vector<DS>(c.n.outputs.size(), c.S(d)), "dim" + std::to_string(d));
  }
  if (linear_in_all_operands) {
    // a sum of partial addends is a partial addend: lets the reduction sink below add/neg/scale/cast
    bool same_shape = true;
    for (int i = 0; i < c.nin(); ++i) same_shape &= c.in(i).numel() == o.numel();
    if (same_shape) c.add(std::vector<DS>(c.nin(), c.P()), std::vector<DS>(c.n.outputs.size(), c.P()), "partial");
  }
  c.add_glue();
}

void SourceRule(Ctx& c) {
  const TensorType& o = c.o();
  if (c.n.op != "constant")
    for (int d = 0; d < o.rank(); ++d)
      if (c.divisible(o, d)) c.add({}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}

// ---- dot family ------------------------------------------------------------------------------
void LinearRule(Ctx& c, const RuleOptions& opt) {
  // y[..,N] = x[..,K] w[N,K]^T (+b[N]) (+res[..,N])
  const TensorType& x = c.in(0);
  const int rx = x.rank();
  const bool has_b = c.n.attr_b("bias"), has_r = c.n.attr_b("residual");
  auto mk = [&](DS xs, DS ws, DS bs, DS rs) {
    std::vector<DS> ins = {xs, ws};
    if (has_b) ins.push_back(bs);
    if (has_r) ins.push_back(rs);
    return ins;
  };
  if (!opt.save_variable_mem)
    for (int d = 0; d < rx - 1; ++d)
      if (c.divisible(x, d)) c.add(mk(c.S(d), c.G(), c.G(), c.S(d)), {c.S(d)}, "batch");
  c.add(mk(c.S(rx - 1), c.S(1), c.G(), c.G()), {c.P()}, "contract");
  // row-parallel with the reduction INSIDE the node as a reduce-scatter over a token dim (Megatron "sequence parallel" form):
  // y_partial = x_s w_s ; y[shard d] = reduce_scatter(y_partial) + b + res[shard d].  The residual stays split -- with the plain
  // "contract" candidate a fused residual has to be replicated, which prices a split residual stream as an all-gather per
  // layer that the rewritten graph never executes.  Cost: the reduce-scatter's bytes (the launch is added by the planner).
  // Opt-in (SpmdOptions::sequence_parallel, strategy "tpsp"): the all-reduce form is what the fused NVLS chains execute and what
  // the tensor-parallel numbers in profiles/ were measured on.
  for (int d = 0; d < rx - 1 && opt.sequence_parallel; ++d)
    if (c.divisible(c.o(), d))
      c.add(mk(c.S(rx - 1), c.S(1), c.G(), c.S(d)), {c.S(d)}, "contract_rs" + std::to_string(d),
            (double)c.o().bytes() * (c.num - 1) / c.num);
  c.add(mk(c.G(), c.S(0), c.S(0), c.S(rx - 1)), {c.S(rx - 1)}, "col");
  if (opt.allow_glue_compute_intensive) c.add_glue();
}
void LinearDgradRule(Ctx& c, const RuleOptions& opt) {
  // dx[..,K] = dy[..,N] w[N,K]
  const TensorType& dy = c.in(0);
  const int r = dy.rank();
  if (!opt.save_variable_mem)
    for (int d = 0; d < r - 1; ++d)
      if (c.divisible(dy, d)) c.add({c.S(d), c.G()}, {c.S(d)}, "batch");
  c.add({c.S(r - 1), c.S(0)}, {c.P()}, "contract");
  c.add({c.G(), c.S(1)}, {c.S(r - 1)}, "col");
  if (opt.allow_glue_compute_intensive) c.add_glue();
}
void LinearWgradRule(Ctx& c, const RuleOptions& opt) {
  // dw[N,K] = dy[..,N]^T x[..,K]  (contraction over all leading dims)
  const TensorType& dy = c.in(0);
  const int r = dy.rank();
  if (!opt.save_variable_mem)
    for (int d = 0; d < r - 1; ++d)
      if (c.divisible(dy, d)) c.add({c.S(d), c.S(d)}, {c.P()}, "contract");
  c.add({c.S(r - 1), c.G()}, {c.S(0)}, "row");
  c.add({c.G(), c.S(r - 1)}, {c.S(1)}, "col");
  if (opt.allow_glue_compute_intensive) c.add_glue();
}
void MatmulRule(Ctx& c, const RuleOptions& opt) {
  const TensorType &a = c.in(0), &b = c.in(1), &o = c.o();
  const bool ta = c.n.attr_b("ta"), tb = c.n.attr_b("tb");
  const int ra = a.rank(), rb = b.rank(), ro = o.rank();
  const int am = ta ? ra - 1 : ra - 2, ak = ta ? ra - 2 : ra - 1;
  const int bk = tb ? rb - 1 : rb - 2, bn = tb ? rb - 2 : rb - 1;
  for (int d = 0; d < ro - 2; ++d) {  // batch dims (leading, right-aligned between operands)
      int da = d - (ro - ra), db = d - (ro - rb);
      DS sa = (da >= 0 && da < ra - 2) ? c.S(da) : c.G();
      DS sb = (db >= 0 && db < rb - 2) ? c.S(db) : c.G();
      if (sa.is_glue() && sb.is_glue()) continue;
      if (opt.save_variable_mem && (sa.is_glue() || sb.is_glue())) continue;
      c.add({sa, sb}, {c.S(d)}, "batch");
    }
  c.add({c.S(ak), c.S(bk)}, {c.P()}, "contract");
  c.add({c.S(am), c.G()}, {c.S(ro - 2)}, "row");
  c.add({c.G(), c.S(bn)}, {c.S(ro - 1)}, "col");
  if (opt.allow_glue_compute_intensive) c.add_glue();
}
void EinsumRule(Ctx& c, const RuleOptions& opt) {
  std::string eq = c.n.attr_s("eq");
  eq.erase(std::remove(eq.begin(), eq.end(), ' '), eq.end());
  auto arrow = eq.find("->");
  std::string lhs = eq.substr(0, arrow), out = eq.substr(arrow + 2);
  auto comma = lhs.find(',');
  std::string ia = lhs.substr(0, comma), ib = lhs.substr(comma + 1);
  std::set<char> labels(lhs.begin(), lhs.end());
  labels.erase(',');
  for (char l : labels) {
    int pa = (int)ia.find(l), pb = (int)ib.find(l), po = (int)out.find(l);
    bool in_a = pa != (int)std::string::npos, in_b = pb != (int)std::string::npos, in_o = po != (int)std::string::npos;
    if (in_a && in_b && in_o) {
      // a batch label shards BOTH operands (e.g. the expert dim of an MoE weight): it never leaves a weight
      // replicated, so the memory-save list does not suppress it (this is how expert parallelism survives)
      c.add({c.S(pa), c.S(pb)}, {c.S(po)}, "batch");
    } else if (in_a && in_b) {
      c.add({c.S(pa), c.S(pb)}, {c.P()}, "contract");
    } else if (in_a && in_o) {
      c.add({c.S(pa), c.G()}, {c.S(po)}, "row");
    } else if (in_b && in_o) {
      c.add({c.G(), c.S(pb)}, {c.S(po)}, "col");
    }
  }
  if (opt.allow_glue_compute_intensive) c.add_glue();
}
void ConvRule(Ctx& c, const RuleOptions& opt) {
  const std::string& op = c.n.op;
  if (op == "conv2d") {  // x[N,C,H,W], w[O,I,kh,kw] -> y[N,O,..]
    if (!opt.save_variable_mem) c.add({c.S(0), c.G()}, {c.S(0)}, "batch");
    c.add({c.S(1), c.S(1)}, {c.P()}, "contract");
    c.add({c.G(), c.S(0)}, {c.S(1)}, "col");
  } else if (op == "conv2d_dgrad") {  // dy[N,O,..], w -> dx[N,C,..]
    if (!opt.save_variable_mem) c.add({c.S(0), c.G()}, {c.S(0)}, "batch");
    c.add({c.S(1), c.S(0)}, {c.P()}, "contract");
    c.add({c.G(), c.S(1)}, {c.S(1)}, "col");
  } else {  // conv2d_wgrad: dy, x -> dw[O,I,kh,kw]
    if (!opt.save_variable_mem) c.add({c.S(0), c.S(0)}, {c.P()}, "contract");
    c.add({c.S(1), c.G()}, {c.S(0)}, "row");
    c.add({c.G(), c.S(1)}, {c.S(1)}, "col");
  }
  if (opt.allow_glue_compute_intensive) c.add_glue();
}

// ---- macro ops -----------------------------------------------------------------------------
void LayerNormRule(Ctx& c) {
  const TensorType& x = c.in(0);
  for (int d = 0; d < x.rank() - 1; ++d)
    if (c.divisible(x, d)) c.add({c.S(d), c.G(), c.G()}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void LayerNormBwdRule(Ctx& c) {
  const TensorType& x = c.in(1);
  for (int d = 0; d < x.rank() - 1; ++d)
    if (c.divisible(x, d)) c.add({c.S(d), c.S(d), c.G()}, {c.S(d), c.P(), c.P()}, "dim" + std::to_string(d));
  c.add_glue();
}
// Context parallelism ("seq" candidates): the sequence stays split through attention; every rank keeps its query block and the
// K / V blocks travel around a ring (causal: blocks from later ranks are skipped, the diagonal block is masked), partial outputs
// merge by log-sum-exp.  The reference has no such op (SURVEY 5.7: long context = token split + what XLA SPMD makes of the dots);
// priced as the K / V all-gather it replaces (forward) plus the dK / dV reduce-scatter (backward).
double RingBytes(const TensorType& qkv, int num) { return (double)qkv.bytes() * (2.0 / 3.0) * (num - 1) / num; }
// Optional document ids (int32 [B, S], the last input; no gradient): they follow qkv's batch split and stay whole along the
// sequence in "seq", so every rank of the ring already holds the key ids of every visiting block and the ring carries no extra
// bytes (ids cost 4 bytes a token against 4 C for the K / V block).  Replicated in "heads" and "glue".
void AttentionRule(Ctx& c, const RuleOptions& opt) {
  // qkv [B,S,H*3*D] (heads-major, so a plain last-dim split is a split over heads) [, segments [B,S]] -> o [B,S,H*D], lse [B,H,S]
  const int64_t H = c.n.attr_i("heads");
  const bool cp = opt.context_parallel && c.divisible(c.in(0), 1);   // "cp": the sequence split is the only way through attention
  auto ins = [&](DS qkv, DS seg) { return c.nin() > 1 ? std::vector<DS>{qkv, seg} : std::vector<DS>{qkv}; };
  if (c.divisible(c.in(0), 0) && !cp) c.add(ins(c.S(0), c.S(0)), {c.S(0), c.S(0)}, "batch");
  if (H % c.num == 0 && !cp) c.add(ins(c.S(2), c.G()), {c.S(2), c.S(1)}, "heads");
  if (c.divisible(c.in(0), 1)) c.add(ins(c.S(1), c.G()), {c.S(1), c.S(2)}, "seq", RingBytes(c.in(0), c.num));
  if (!cp) c.add_glue();   // (replicated attention = n x the S^2 FLOPs per rank: never what "cp" asks for)
}
void AttentionBwdRule(Ctx& c, const RuleOptions& opt) {
  const int64_t H = c.n.attr_i("heads");  // (do, qkv, o, lse [, segments]) -> dqkv
  const bool cp = opt.context_parallel && c.divisible(c.in(1), 1);
  auto ins = [&](std::vector<DS> v, DS seg) { if (c.nin() > 4) v.push_back(seg); return v; };
  if (c.divisible(c.in(1), 0) && !cp) c.add(ins({c.S(0), c.S(0), c.S(0), c.S(0)}, c.S(0)), {c.S(0)}, "batch");
  if (H % c.num == 0 && !cp) c.add(ins({c.S(2), c.S(2), c.S(2), c.S(1)}, c.G()), {c.S(2)}, "heads");
  if (c.divisible(c.in(1), 1)) c.add(ins({c.S(1), c.S(1), c.S(1), c.S(2)}, c.G()), {c.S(1)}, "seq", 2.0 * RingBytes(c.in(1), c.num));
  if (!cp) c.add_glue();
}
void EmbeddingRule(Ctx& c) {  // tokens[B,S], wte[V,C], wpe[S,C] -> [B,S,C]
  if (c.divisible(c.in(0), 0)) c.add({c.S(0), c.G(), c.G()}, {c.S(0)}, "batch");
  // sequence split: rank r embeds positions [r S/n, (r+1) S/n) -- exactly the rows of a position table stored split on dim 0
  if (c.divisible(c.in(0), 1) && c.in(2).dims[0] == c.in(0).dims[1]) c.add({c.S(1), c.G(), c.S(0)}, {c.S(1)}, "seq");
  c.add({c.G(), c.S(1), c.S(1)}, {c.S(2)}, "hidden");
  c.add_glue();
}
void EmbeddingBwdRule(Ctx& c) {  // tokens, dy[B,S,C] -> dwte[V,C], dwpe[S,C]
  if (c.divisible(c.in(0), 0)) c.add({c.S(0), c.S(0)}, {c.P(), c.P()}, "batch");
  if (c.divisible(c.in(0), 1) && c.o(1).dims[0] == c.in(0).dims[1]) c.add({c.S(1), c.S(1)}, {c.P(), c.S(0)}, "seq");
  c.add({c.G(), c.S(2)}, {c.S(1), c.S(1)}, "hidden");
  c.add_glue();
}
void XentRule(Ctx& c) {  // logits[..,V], labels[..] -> loss[], dlogits
  const TensorType& l = c.in(0);
  for (int d = 0; d < l.rank() - 1; ++d)
    if (c.divisible(l, d)) c.add({c.S(d), c.S(d)}, {c.P(), c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void ColsumRule(Ctx& c) {
  const TensorType& x = c.in(0);
  for (int d = 0; d < x.rank() - 1; ++d)
    if (c.divisible(x, d)) c.add({c.S(d)}, {c.P()}, "dim" + std::to_string(d));
  c.add({c.S(x.rank() - 1)}, {c.S(0)}, "last");
  c.add_glue();
}
void ReduceRule(Ctx& c) {
  const TensorType& x = c.in(0);
  auto axes = c.n.attr_v("axes");
  const bool keep = c.n.attr_b("keepdims");
  const int kind = c.n.op == "reduce_max" ? 1 : 0;
  for (int d = 0; d < x.rank(); ++d) {
    if (!c.divisible(x, d)) continue;
    if (std::find(axes.begin(), axes.end(), (int64_t)d) != axes.end()) {
      c.add({c.S(d)}, {c.P(kind)}, "reduced");
    } else {
      int od = d;
      if (!keep)
        for (auto a : axes)
          if (a < d) --od;
      c.add({c.S(d)}, {c.S(od)}, "dim" + std::to_string(d));
    }
  }
  c.add_glue();
}
void BroadcastRule(Ctx& c) {
  auto dims = c.n.attr_v("dims");
  const TensorType& o = c.o();
  for (int d = 0; d < o.rank(); ++d) {
    if (!c.divisible(o, d)) continue;
    auto it = std::find(dims.begin(), dims.end(), (int64_t)d);
    DS xs = it == dims.end() ? c.G() : c.S((int)(it - dims.begin()));
    c.add({xs}, {c.S(d)}, "dim" + std::to_string(d));
  }
  c.add_glue();
}
void ReshapeRule(Ctx& c) {
  const TensorType &x = c.in(0), &o = c.o();
  std::set<std::pair<DS, DS>> seen;
  for (int d = 0; d < x.rank(); ++d) {
    if (!c.divisible(x, d)) continue;
    DS xs = c.S(d), os = xs.ApplyToShape(x, o);
    if (os.is_glue() || !os.Valid(o)) continue;
    if (seen.insert({xs, os}).second) c.add({xs}, {os}, "in" + std::to_string(d));
  }
  for (int d = 0; d < o.rank(); ++d) {
    if (!c.divisible(o, d)) continue;
    DS os = c.S(d), xs = os.ApplyToShape(o, x);
    if (xs.is_glue() || !xs.Valid(x)) continue;
    if (seen.insert({xs, os}).second) c.add({xs}, {os}, "out" + std::to_string(d));
  }
  c.add({c.P()}, {c.P()}, "partial");
  c.add_glue();
}
void TransposeRule(Ctx& c) {
  auto perm = c.n.attr_v("perm");
  const TensorType& o = c.o();
  for (int d = 0; d < o.rank(); ++d)
    if (c.divisible(o, d)) c.add({c.S((int)perm[d])}, {c.S(d)}, "dim" + std::to_string(d));
  c.add({c.P()}, {c.P()}, "partial");
  c.add_glue();
}
void SliceRule(Ctx& c) {
  const TensorType &x = c.in(0), &o = c.o();
  for (int d = 0; d < x.rank(); ++d)  // only dims the slice fully covers (reference InferSlice, utils.cc:428-447)
    if (x.dims[d] == o.dims[d] && c.divisible(x, d)) c.add({c.S(d)}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void ConcatRule(Ctx& c) {
  const int axis = (int)c.n.attr_i("axis");
  const TensorType& o = c.o();
  for (int d = 0; d < o.rank(); ++d)
    if (d != axis && c.divisible(o, d)) c.add(std::vector<DS>(c.nin(), c.S(d)), {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void SoftmaxRule(Ctx& c) {
  const int axis = (int)c.n.attr_i("axis");
  const TensorType& o = c.o();
  for (int d = 0; d < o.rank(); ++d)
    if (d != axis && c.divisible(o, d)) c.add(std::vector<DS>(c.nin(), c.S(d)), {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void GatherRule(Ctx& c) {  // table[V, ...], idx[...] -> [idx..., table[1:]...]
  const TensorType &t = c.in(0), &idx = c.in(1);
  for (int d = 0; d < idx.rank(); ++d)
    if (c.divisible(idx, d)) c.add({c.G(), c.S(d)}, {c.S(d)}, "index");
  for (int d = 1; d < t.rank(); ++d)
    if (c.divisible(t, d)) c.add({c.S(d), c.G()}, {c.S(idx.rank() + d - 1)}, "slice");
  c.add_glue();
}
void ScatterAddRule(Ctx& c) {  // idx[...], dy[..., C] -> table grad [V, C]
  const TensorType &idx = c.in(0), &dy = c.in(1);
  for (int d = 0; d < idx.rank(); ++d)
    if (c.divisible(idx, d)) c.add({c.S(d), c.S(d)}, {c.P()}, "index");
  c.add({c.G(), c.S(dy.rank() - 1)}, {c.S(1)}, "slice");
  c.add_glue();
}
void OneHotRule(Ctx& c) {
  const TensorType& idx = c.in(0);
  for (int d = 0; d < idx.rank(); ++d)
    if (c.divisible(idx, d)) c.add({c.S(d)}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void BatchNormRule(Ctx& c) {  // x[N,C,H,W], g[C], b[C]
  const double stat_bytes = 2.0 * 4.0 * (double)c.in(0).dims[1];
  c.add({c.S(0), c.G(), c.G()}, {c.S(0)}, "batch", 2.0 * stat_bytes);  // cross-replica statistics (sync BN)
  c.add({c.S(1), c.S(0), c.S(0)}, {c.S(1)}, "channel");
  c.add_glue();
}
void BatchNormBwdRule(Ctx& c) {  // dy, x, g -> dx, dg, db
  const double stat_bytes = 2.0 * 4.0 * (double)c.in(0).dims[1];
  c.add({c.S(0), c.S(0), c.G()}, {c.S(0), c.P(), c.P()}, "batch", 2.0 * stat_bytes);
  c.add({c.S(1), c.S(1), c.S(0)}, {c.S(1), c.S(0), c.S(0)}, "channel");
  c.add_glue();
}
void Pool4dRule(Ctx& c) {  // any op whose operands/outputs all carry [N, C, ...] : split N or C
  for (int d = 0; d < 2; ++d) {
    bool ok = true;
    for (int i = 0; i < c.nin(); ++i) ok &= c.divisible(c.in(i), d);
    ok &= c.divisible(c.o(), d);
    if (ok) c.add(std::vector<DS>(c.nin(), c.S(d)), {c.S(d)}, "dim" + std::to_string(d));
  }
  c.add_glue();
}
void PadZeroRule(Ctx& c) {
  const TensorType &x = c.in(0), &o = c.o();
  for (int d = 0; d < x.rank(); ++d)
    if (x.dims[d] == o.dims[d] && c.divisible(x, d)) c.add({c.S(d)}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void ApplyRule(Ctx& c) {  // optimizer update: every operand / output shares the variable's layout
  const TensorType& p = c.in(0);
  for (int d = 0; d < p.rank(); ++d)
    if (c.divisible(p, d)) c.add(std::vector<DS>(c.nin(), c.S(d)), std::vector<DS>(c.n.outputs.size(), c.S(d)), "dim" + std::to_string(d));
  c.add_glue();
}

// Optimizers with reduced-shape slots.  The variable (and gradient, and full-shaped slots) may be split on any dim d; a slot
// that keeps dim d is split along with it, a slot that has reduced dim d away is replicated -- its reduction over d is then
// completed across the shards by the executor (an all-reduce of a small vector), which is why these stay single nodes
// instead of being expanded into primitive reductions.
void AdafactorRule(Ctx& c) {
  // (p, g, vr [..., R], vc [..., C]) for p [..., R, C], or (p, g, vf) un-factored
  const TensorType& p = c.in(0);
  const int r = p.rank();
  const bool factored = c.nin() == 4;
  for (int d = 0; d < r; ++d) {
    if (!c.divisible(p, d)) continue;
    std::vector<DS> st;
    if (!factored) st = {c.S(d)};
    else st = {d == r - 1 ? c.G() : c.S(d), d == r - 2 ? c.G() : (d == r - 1 ? c.S(r - 2) : c.S(d))};
    std::vector<DS> ins = {c.S(d), c.S(d)}, outs = {c.S(d)};
    for (auto& x : st) ins.push_back(x), outs.push_back(x);
    c.add(ins, outs, "dim" + std::to_string(d));
  }
  c.add_glue();
}
void Sm3Rule(Ctx& c) {
  // (p, g, acc_0 [d0], ..., acc_{r-1} [d_{r-1}] [, mom]) for rank >= 2; (p, g, acc [, mom]) with a full-shaped acc otherwise
  const TensorType& p = c.in(0);
  const int r = p.rank();
  for (int d = 0; d < r; ++d) {
    if (!c.divisible(p, d)) continue;
    std::vector<DS> ins = {c.S(d), c.S(d)}, outs = {c.S(d)};
    for (int i = 2; i < c.nin(); ++i) {
      const TensorType& t = c.in(i);
      DS x = t.rank() == r ? c.S(d) : (i - 2 == d ? c.S(0) : c.G());   // full-shaped (acc of a vector, momentum) or per-dim
      ins.push_back(x);
      outs.push_back(x);
    }
    c.add(ins, outs, "dim" + std::to_string(d));
  }
  c.add_glue();
}

// ---- ops a traced torch / HLO-like graph brings along (reference: P/utils.cc:598-612 reverse, :734-917 pad / reduce-window /
// select-and-scatter / sort / scatter, :1955-1981 iota) -----------------------------------------------------------------------
void AxesUntouchedRule(Ctx& c, const std::vector<int64_t>& touched) {
  // every operand and output has the input's rank; dims the op does NOT act along can be split on all of them at once
  const TensorType& x = c.nin() ? c.in(0) : c.o();
  for (int d = 0; d < x.rank(); ++d) {
    if (std::find(touched.begin(), touched.end(), (int64_t)d) != touched.end()) continue;
    bool ok = c.divisible(c.o(), d);
    for (int i = 0; i < c.nin(); ++i) ok &= c.in(i).rank() == x.rank() && c.divisible(c.in(i), d);
    if (ok) c.add(std::vector<DS>(c.nin(), c.S(d)), std::vector<DS>(c.n.outputs.size(), c.S(d)), "dim" + std::to_string(d));
  }
  c.add_glue();
}
void ReverseRule(Ctx& c) { AxesUntouchedRule(c, c.n.attr_v("dims")); }          // a reversed dim would need a shard permutation
void SortRule(Ctx& c) { AxesUntouchedRule(c, {c.n.attr_i("axis", -1) < 0 ? c.in(0).rank() + c.n.attr_i("axis", -1) : c.n.attr_i("axis")}); }
void WindowRule(Ctx& c) {
  // reduce_window (x) / select_and_scatter (x, source): a dim is local iff its window is 1 wide, stride 1 and unpadded
  const TensorType& x = c.in(0);
  auto win = c.n.attr_v("window"), str = c.n.attr_v("strides"), pad = c.n.attr_v("padding");
  std::vector<int64_t> touched;
  for (int d = 0; d < x.rank(); ++d) {
    const int64_t w = d < (int)win.size() ? win[d] : 1, s_ = d < (int)str.size() ? str[d] : 1;
    const int64_t p0 = 2 * d < (int)pad.size() ? pad[2 * d] : 0, p1 = 2 * d + 1 < (int)pad.size() ? pad[2 * d + 1] : 0;
    if (w != 1 || s_ != 1 || p0 != 0 || p1 != 0) touched.push_back(d);
  }
  AxesUntouchedRule(c, touched);
}
void PadRule(Ctx& c) {
  // general pad (low / high / interior per dim): dims that are not padded keep their split
  const TensorType& x = c.in(0);
  auto lo = c.n.attr_v("low"), hi = c.n.attr_v("high"), in_ = c.n.attr_v("interior");
  for (int d = 0; d < x.rank(); ++d) {
    const bool padded = (d < (int)lo.size() && lo[d]) || (d < (int)hi.size() && hi[d]) || (d < (int)in_.size() && in_[d]);
    if (padded || !c.divisible(x, d) || !c.divisible(c.o(), d)) continue;
    std::vector<DS> ins(c.nin(), c.G());    // (operand 1, when present, is the scalar padding value)
    ins[0] = c.S(d);
    c.add(ins, {c.S(d)}, "dim" + std::to_string(d));
  }
  c.add_glue();
}
void IotaRule(Ctx& c) {
  // source: shards along a non-iota dim are identical copies; the iota dim itself would need a per-shard offset
  const TensorType& o = c.o();
  const int64_t id = c.n.attr_i("dim", 0);
  for (int d = 0; d < o.rank(); ++d)
    if (d != id && c.divisible(o, d)) c.add({}, {c.S(d)}, "dim" + std::to_string(d));
  c.add_glue();
}
void SelectRule(Ctx& c) { Elementwise(c, false); }   // select(pred, a, b) / clamp(lo, x, hi): broadcast-aware elementwise
void ScatterRule(Ctx& c) {
  // scatter(operand, indices, updates) along `axis`: every other dim of operand / updates (and of equally shaped indices) is local
  const TensorType& x = c.in(0);
  int64_t ax = c.n.attr_i("axis", 0);
  if (ax < 0) ax += x.rank();
  for (int d = 0; d < x.rank(); ++d) {
    if (d == ax || !c.divisible(x, d) || !c.divisible(c.o(), d)) continue;
    std::vector<DS> ins = {c.S(d)};
    bool ok = true;
    for (int i = 1; i < c.nin(); ++i) {
      if (c.in(i).rank() == x.rank() && c.divisible(c.in(i), d)) ins.push_back(c.S(d));
      else ok = false;
    }
    if (ok) c.add(ins, {c.S(d)}, "dim" + std::to_string(d));
  }
  c.add_glue();
}

std::set<std::string>& UnknownOpsSeen() {
  static std::set<std::string> s;
  return s;
}

}  // namespace

std::vector<Candidate> EnumerateCandidates(const Graph& g, const Node& n, int num, const RuleOptions& opt) {
  Ctx c{g, n, num, {}};
  const std::string& op = n.op;
  static const std::set<std::string> unary_linear = {"neg", "scale", "cast"};
  static const std::set<std::string> unary = {"gelu", "relu", "tanh", "exp", "log", "sqrt", "rsqrt", "sigmoid", "abs", "sign", "erf",
                                               "logical_not", "floor", "ceil", "silu"};
  static const std::set<std::string> binary_linear = {"add", "sub"};
  static const std::set<std::string> binary = {"mul", "div", "relu_bwd", "tanh_bwd", "gelu_bwd", "maximum", "minimum", "pow", "compare",
                                                "logical_and", "logical_or", "sigmoid_bwd", "silu_bwd"};
  if (IsSource(op)) SourceRule(c);
  else if (unary_linear.count(op) || binary_linear.count(op)) Elementwise(c, true);
  else if (unary.count(op) || binary.count(op)) Elementwise(c, false);
  else if (op == "linear") LinearRule(c, opt);
  else if (op == "linear_dgrad") LinearDgradRule(c, opt);
  else if (op == "linear_wgrad") LinearWgradRule(c, opt);
  else if (op == "matmul") MatmulRule(c, opt);
  else if (op == "einsum") EinsumRule(c, opt);
  else if (op == "conv2d" || op == "conv2d_dgrad" || op == "conv2d_wgrad") ConvRule(c, opt);
  else if (op == "layernorm") LayerNormRule(c);
  else if (op == "layernorm_bwd") LayerNormBwdRule(c);
  else if (op == "attention") AttentionRule(c, opt);
  else if (op == "attention_bwd") AttentionBwdRule(c, opt);
  else if (op == "embedding") EmbeddingRule(c);
  else if (op == "embedding_bwd") EmbeddingBwdRule(c);
  else if (op == "softmax_xent") XentRule(c);
  else if (op == "colsum") ColsumRule(c);
  else if (op == "reduce_sum" || op == "reduce_mean" || op == "reduce_max") ReduceRule(c);
  else if (op == "broadcast") BroadcastRule(c);
  else if (op == "reshape") ReshapeRule(c);
  else if (op == "transpose") TransposeRule(c);
  else if (op == "slice") SliceRule(c);
  else if (op == "pad_zero") PadZeroRule(c);
  else if (op == "concat") ConcatRule(c);
  else if (op == "softmax" || op == "softmax_bwd") SoftmaxRule(c);
  else if (op == "gather") GatherRule(c);
  else if (op == "scatter_add") ScatterAddRule(c);
  else if (op == "one_hot") OneHotRule(c);
  else if (op == "batchnorm") BatchNormRule(c);
  else if (op == "batchnorm_bwd") BatchNormBwdRule(c);
  else if (op == "maxpool2d" || op == "maxpool2d_bwd" || op == "global_avgpool" || op == "global_avgpool_bwd") Pool4dRule(c);
  else if (op == "apply_adamw" || op == "apply_sgd" || op == "apply_momentum" || op == "apply_lamb") ApplyRule(c);
  else if (op == "apply_adafactor") AdafactorRule(c);
  else if (op == "apply_sm3") Sm3Rule(c);
  else if (op == "moe_dispatch_mask" || op == "moe_dispatch_mask_bwd") {  // gating is independent per token group
    bool ok = true;
    for (int i = 0; i < c.nin(); ++i) ok &= c.divisible(c.in(i), 0);
    if (ok) c.add(std::vector<DS>(c.nin(), c.S(0)), {c.S(0)}, "group");
    c.add_glue();
  }
  else if (op == "reverse") ReverseRule(c);
  else if (op == "sort") SortRule(c);
  else if (op == "reduce_window" || op == "select_and_scatter") WindowRule(c);
  else if (op == "pad") PadRule(c);
  else if (op == "iota") IotaRule(c);
  else if (op == "select" || op == "clamp") SelectRule(c);
  else if (op == "scatter") ScatterRule(c);
  else {
    UnknownOpsSeen().insert(op);   // replicated only (safe) -- but never silently: the planner reports these (SpmdStats.unknown_ops)
    c.add_glue();
  }
  return std::move(c.out);
}

std::vector<Candidate> ForwardInfer(const Graph& g, const Node& n, int num, int operand_idx, const DimStrategy& s) {
  RuleOptions opt;
  opt.allow_glue_compute_intensive = true;
  std::vector<Candidate> r;
  for (auto& c : EnumerateCandidates(g, n, num, opt))
    if (operand_idx < (int)c.ins.size() && c.ins[operand_idx] == s) r.push_back(c);
  return r;
}
std::vector<Candidate> BackInfer(const Graph& g, const Node& n, int num, int out_idx, const DimStrategy& s) {
  RuleOptions opt;
  opt.allow_glue_compute_intensive = true;
  std::vector<Candidate> r;
  for (auto& c : EnumerateCandidates(g, n, num, opt))
    if (out_idx < (int)c.outs.size() && c.outs[out_idx] == s) r.push_back(c);
  return r;
}

TensorType ShardType(const TensorType& t, const DimStrategy& s) {
  TensorType r = t;
  if (s.is_split()) r.dims[s.dim] /= s.num;
  return r;
}

bool InferGraph(const Graph& g, int num, std::map<ValueRef, DimStrategy>* assign, std::string* conflict) {
  RuleOptions opt;
  opt.allow_glue_compute_intensive = true;
  std::vector<std::vector<Candidate>> cands(g.nodes.size());
  for (auto& n : g.nodes) cands[n.id] = EnumerateCandidates(g, n, num, opt);
  bool changed = true;
  int sweeps = 0;
  while (changed && sweeps++ < 64) {
    changed = false;
    auto visit = [&](const Node& n) -> bool {
      // candidates consistent with everything already assigned around this node
      std::vector<const Candidate*> ok;
      bool any_assigned = false;
      for (auto& c : cands[n.id]) {
        bool good = true;
        for (int i = 0; i < (int)n.inputs.size() && good; ++i) {
          auto it = assign->find(n.inputs[i]);
          if (it == assign->end()) continue;
          any_assigned = true;
          // a partial producer is reduced before use; a replicated producer can be sliced for free
          if (it->second.partial || it->second.is_glue()) continue;
          if (c.ins[i] != it->second) good = false;
        }
        for (int o = 0; o < (int)n.outputs.size() && good; ++o) {
          auto it = assign->find(ValueRef{n.id, o});
          if (it == assign->end()) continue;
          any_assigned = true;
          if (c.outs[o] != it->second) good = false;
        }
        if (good) ok.push_back(&c);
      }
      if (!any_assigned) return true;
      if (ok.empty()) {
        if (conflict) *conflict = n.name + " (" + n.op + ")";
        return false;
      }
      // prefer non-glue candidates that are forced by a split neighbour
      std::vector<const Candidate*> pref;
      for (auto* c : ok) {
        bool touches_split = false;
        for (int i = 0; i < (int)n.inputs.size(); ++i) {
          auto it = assign->find(n.inputs[i]);
          if (it != assign->end() && it->second.is_split() && c->ins[i] == it->second) touches_split = true;
        }
        for (int o = 0; o < (int)n.outputs.size(); ++o) {
          auto it = assign->find(ValueRef{n.id, o});
          if (it != assign->end() && it->second.is_split() && c->outs[o] == it->second) touches_split = true;
        }
        if (touches_split) pref.push_back(c);
      }
      if (pref.empty()) return true;
      // assign whatever all preferred candidates agree on
      for (int o = 0; o < (int)n.outputs.size(); ++o) {
        ValueRef v{n.id, o};
        if (assign->count(v)) continue;
        bool agree = true;
        for (auto* c : pref) agree &= (c->outs[o] == pref[0]->outs[o]);
        if (agree) { (*assign)[v] = pref[0]->outs[o]; changed = true; }
      }
      for (int i = 0; i < (int)n.inputs.size(); ++i) {
        if (assign->count(n.inputs[i])) continue;
        bool agree = true;
        for (auto* c : pref) agree &= (c->ins[i] == pref[0]->ins[i]);
        if (agree && !pref[0]->ins[i].is_glue()) { (*assign)[n.inputs[i]] = pref[0]->ins[i]; changed = true; }
      }
      return true;
    };
    for (auto& n : g.nodes)
      if (!visit(n)) return false;
    for (auto it = g.nodes.rbegin(); it != g.nodes.rend(); ++it)
      if (!visit(*it)) return false;
  }
  return true;
}

std::vector<std::string> UnknownOps(bool clear) {
  std::vector<std::string> r(UnknownOpsSeen().begin(), UnknownOpsSeen().end());
  if (clear) UnknownOpsSeen().clear();
  return r;
}

// Round-trip check of the rule table on a whole graph (reference VerifyInfer, P/utils.cc:1781-1848): for every node and every
// candidate, (1) every split divides its dimension, (2) re-deriving the candidate from any single operand layout (ForwardInfer)
// or output layout (BackInfer) finds it again, (3) the shard shapes are what the op would produce from its shard operands for
// the shape-preserving op families (elementwise: output shard dims == broadcast of operand shard dims).  Returns violations.
std::vector<std::string> VerifyInfer(const Graph& g, int num) {
  std::vector<std::string> bad;
  RuleOptions opt;
  opt.allow_glue_compute_intensive = true;
  auto same = [](const Candidate& a, const Candidate& b) { return a.ins == b.ins && a.outs == b.outs; };
  for (const auto& n : g.nodes) {
    auto cands = EnumerateCandidates(g, n, num, opt);
    if (cands.empty()) bad.push_back(n.op + " '" + n.name + "': no candidate at all");
    for (const auto& c : cands) {
      if (c.ins.size() != n.inputs.size() || c.outs.size() != n.outputs.size()) {
        bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: arity mismatch");
        continue;
      }
      for (size_t i = 0; i < c.ins.size(); ++i) {
        if (c.ins[i].is_split() && !c.ins[i].Valid(g.type(n.inputs[i])))
          bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: operand " + std::to_string(i) + " split does not divide");
        bool found = false;
        for (const auto& f : ForwardInfer(g, n, num, (int)i, c.ins[i])) found |= same(f, c);
        if (!found) bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: forward round trip from operand " + std::to_string(i) + " lost it");
      }
      for (size_t j = 0; j < c.outs.size(); ++j) {
        if (c.outs[j].is_split() && !c.outs[j].Valid(n.outputs[j]))
          bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: output " + std::to_string(j) + " split does not divide");
        bool found = false;
        for (const auto& f : BackInfer(g, n, num, (int)j, c.outs[j])) found |= same(f, c);
        if (!found) bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: backward round trip from output " + std::to_string(j) + " lost it");
      }
      // shape algebra for elementwise families: out shard dim == max over operand shard dims (right-aligned broadcasting)
      static const std::set<std::string> ew = {"add", "sub", "mul", "div", "neg", "scale", "cast", "gelu", "relu", "tanh", "exp", "log",
                                               "maximum", "minimum", "select", "clamp", "sqrt", "rsqrt", "sigmoid", "abs"};
      if (ew.count(n.op) && !c.outs.empty() && !c.outs[0].partial) {
        TensorType so = ShardType(n.outputs[0], c.outs[0]);
        for (size_t i = 0; i < c.ins.size(); ++i) {
          if (c.ins[i].partial) continue;
          TensorType si = ShardType(g.type(n.inputs[i]), c.ins[i]);
          const int off = so.rank() - si.rank();
          for (int d = 0; d < si.rank(); ++d)
            if (si.dims[d] != 1 && si.dims[d] != so.dims[d + off])
              bad.push_back(n.op + " '" + n.name + "' [" + c.tag + "]: shard shapes of operand " + std::to_string(i) + " and output disagree");
        }
      }
    }
  }
  return bad;
}

}  // namespace tepdist
