#include "ir.h"

#include <algorithm>
#include <set>
#include <sstream>

namespace tepdist {

std::string DimStrategy::str() const {
  std::ostringstream o;
  if (partial) {
    o << "P(" << num << ")";
  } else if (dim < 0) {
    o << "G";
  } else {
    o << "S(" << dim << "/" << num;
    if (stride > 0) o << ",stride=" << stride;
    o << ")";
  }
  return o.str();
}

bool DimStrategy::Valid(const TensorType& t) const {
  if (!is_split()) return true;
  if (dim >= t.rank()) return false;
  int64_t s = EffStride(t);
  if (s <= 0 || t.dims[dim] % s != 0) return false;
  return s % num == 0;
}

int64_t DimStrategy::StrideOnElements(const TensorType& t) const {
  int64_t e = EffStride(t);
  for (int i = dim + 1; i < t.rank(); ++i) e *= t.dims[i];
  return e;
}

DimStrategy DimStrategy::ApplyToShape(const TensorType& from, const TensorType& to) const {
  if (!is_split()) return *this;
  if (from.numel() != to.numel()) return Glue();
  // One period of the split covers `soe` consecutive row-major elements; each shard owns a contiguous
  // soe/num chunk of every period.  Find the dim of `to` whose suffix product reaches `soe`.
  const int64_t soe = StrideOnElements(from);
  int64_t acc = 1;
  for (int d = to.rank() - 1; d >= 0; --d) {
    const int64_t below = acc;  // elements to the right of dim d
    acc *= to.dims[d];
    if (acc >= soe) {
      if (soe % below != 0) return Glue();
      const int64_t stride = soe / below;  // period length measured along dim d
      if (stride <= 0 || to.dims[d] % stride != 0 || stride % num != 0) return Glue();
      // the shard chunk must be a whole number of rows of the dims to the right
      if ((soe / num) % below != 0) return Glue();
      DimStrategy r = Split(d, num, stride == to.dims[d] ? 0 : stride);
      return r;
    }
  }
  return Glue();
}

std::string DistSpec::str() const {
  std::ostringstream o;
  o << "[";
  for (size_t i = 0; i < levels.size(); ++i) o << (i ? "," : "") << levels[i].str();
  o << "]";
  if (stage >= 0) o << "@" << stage;
  return o.str();
}

int64_t Node::attr_i(const std::string& k, int64_t def) const {
  auto it = attrs.find(k);
  if (it == attrs.end()) return def;
  if (auto p = std::get_if<int64_t>(&it->second)) return *p;
  if (auto p = std::get_if<bool>(&it->second)) return *p ? 1 : 0;
  if (auto p = std::get_if<double>(&it->second)) return (int64_t)*p;
  return def;
}
double Node::attr_f(const std::string& k, double def) const {
  auto it = attrs.find(k);
  if (it == attrs.end()) return def;
  if (auto p = std::get_if<double>(&it->second)) return *p;
  if (auto p = std::get_if<int64_t>(&it->second)) return (double)*p;
  return def;
}
bool Node::attr_b(const std::string& k, bool def) const {
  auto it = attrs.find(k);
  if (it == attrs.end()) return def;
  if (auto p = std::get_if<bool>(&it->second)) return *p;
  if (auto p = std::get_if<int64_t>(&it->second)) return *p != 0;
  return def;
}
std::string Node::attr_s(const std::string& k, const std::string& def) const {
  auto it = attrs.find(k);
  if (it == attrs.end()) return def;
  if (auto p = std::get_if<std::string>(&it->second)) return *p;
  return def;
}
std::vector<int64_t> Node::attr_v(const std::string& k) const {
  auto it = attrs.find(k);
  if (it == attrs.end()) return {};
  if (auto p = std::get_if<std::vector<int64_t>>(&it->second)) return *p;
  return {};
}

int Graph::AddNode(const std::string& op, const std::vector<ValueRef>& inputs, const std::vector<TensorType>& outs,
                   const std::map<std::string, Attr>& attrs, const std::string& name, int group, bool backward) {
  Node n;
  n.id = (int)nodes.size();
  n.op = op;
  n.inputs = inputs;
  n.outputs = outs;
  n.attrs = attrs;
  n.name = name.empty() ? op + "_" + std::to_string(n.id) : name;
  n.group = group;
  n.backward = backward;
  n.dist.resize(outs.size());
  nodes.push_back(std::move(n));
  users_valid_ = false;
  return nodes.back().id;
}

const std::vector<Use>& Graph::users(ValueRef v) const {
  if (!users_valid_) {
    users_.clear();
    for (const auto& n : nodes)
      for (int i = 0; i < (int)n.inputs.size(); ++i) users_[n.inputs[i]].push_back({n.id, i});
    users_valid_ = true;
  }
  auto it = users_.find(v);
  return it == users_.end() ? empty_ : it->second;
}

std::string Graph::Dump(bool with_dist) const {
  std::ostringstream o;
  o << "graph " << name << " split_nums=[";
  for (size_t i = 0; i < split_nums.size(); ++i) o << (i ? "," : "") << split_nums[i] << (share_dev[i] ? "t" : "");
  o << "]\n";
  for (const auto& n : nodes) {
    o << "  %" << n.id << " = " << n.op << "(";
    for (size_t i = 0; i < n.inputs.size(); ++i) {
      o << (i ? ", " : "") << "%" << n.inputs[i].node;
      if (n.inputs[i].idx) o << "." << n.inputs[i].idx;
    }
    o << ") -> ";
    for (size_t i = 0; i < n.outputs.size(); ++i) {
      o << (i ? ", " : "") << n.outputs[i].dtype << "[";
      for (size_t d = 0; d < n.outputs[i].dims.size(); ++d) o << (d ? "," : "") << n.outputs[i].dims[d];
      o << "]";
      if (with_dist && i < n.dist.size() && !n.dist[i].levels.empty()) o << n.dist[i].str();
    }
    o << "  # " << n.name << " g=" << n.group << (n.backward ? " bwd" : "");
    if (n.stage >= 0) o << " stage=" << n.stage;
    o << "\n";
  }
  return o.str();
}

bool IsSource(const std::string& op) {
  return op == "parameter" || op == "input" || op == "constant" || op == "state";
}
bool IsVariable(const std::string& op) { return op == "parameter" || op == "state"; }
bool IsComputeIntensive(const std::string& op) {
  static const std::set<std::string> s = {"linear", "linear_dgrad", "linear_wgrad", "matmul", "einsum", "conv2d",
                                          "conv2d_dgrad", "conv2d_wgrad"};
  return s.count(op) > 0;
}
bool IsCollective(const std::string& op) {
  static const std::set<std::string> s = {"all_reduce", "all_gather", "reduce_scatter", "all_to_all",
                                          "dynamic_slice", "send", "recv"};
  return s.count(op) > 0;
}

double NodeFlops(const Graph& g, const Node& n) {
  auto numel = [&](ValueRef v) { return (double)g.type(v).numel(); };
  const std::string& op = n.op;
  if (op == "linear" || op == "linear_dgrad") {
    // out[..,N] over contraction K: 2 * numel(out) * K
    const TensorType& w = g.type(n.inputs[1]);
    double k = op == "linear" ? (double)w.dims[1] : (double)w.dims[0];
    return 2.0 * (double)n.outputs[0].numel() * k;
  }
  if (op == "linear_wgrad") {
    const TensorType& dy = g.type(n.inputs[0]);
    double tokens = (double)dy.numel() / (double)dy.dims.back();
    return 2.0 * (double)n.outputs[0].numel() * tokens;
  }
  if (op == "matmul") {
    const TensorType& a = g.type(n.inputs[0]);
    double k = n.attr_b("ta") ? (double)a.dims[a.rank() - 2] : (double)a.dims[a.rank() - 1];
    return 2.0 * (double)n.outputs[0].numel() * k;
  }
  if (op == "einsum") {
    // contraction size = numel(a) * numel(b) / (numel(out) * batch^2...) -> derive from the equation
    std::string eq = n.attr_s("eq");
    auto arrow = eq.find("->");
    std::string lhs = eq.substr(0, arrow), out = eq.substr(arrow + 2);
    auto comma = lhs.find(',');
    std::string ia = lhs.substr(0, comma), ib = lhs.substr(comma + 1);
    std::map<char, int64_t> dims;
    const TensorType& a = g.type(n.inputs[0]);
    const TensorType& b = g.type(n.inputs[1]);
    for (size_t i = 0; i < ia.size(); ++i) dims[ia[i]] = a.dims[i];
    for (size_t i = 0; i < ib.size(); ++i) dims[ib[i]] = b.dims[i];
    double f = 2.0;
    for (auto& kv : dims) f *= (double)kv.second;
    return f;
  }
  if (op == "conv2d" || op == "conv2d_dgrad" || op == "conv2d_wgrad") {
    // 2 * numel(y) * C_in * kh * kw
    const TensorType* w = nullptr;
    const TensorType* y = nullptr;
    if (op == "conv2d") { w = &g.type(n.inputs[1]); y = &n.outputs[0]; }
    else if (op == "conv2d_dgrad") { w = &g.type(n.inputs[1]); y = &g.type(n.inputs[0]); }
    else { w = &n.outputs[0]; y = &g.type(n.inputs[0]); }
    return 2.0 * (double)y->numel() * (double)(w->dims[1] * w->dims[2] * w->dims[3]);
  }
  // Attention FLOPs stay the causal / full count with document masking too: document lengths are only known from the data.
  if (op == "attention") {
    const TensorType& qkv = g.type(n.inputs[0]);
    double B = qkv.dims[0], S = qkv.dims[1], C = qkv.dims[2] / 3.0;
    double f = 4.0 * B * S * S * C;
    return n.attr_b("causal", true) ? f / 2 : f;
  }
  if (op == "attention_bwd") {
    const TensorType& qkv = g.type(n.inputs[1]);
    double B = qkv.dims[0], S = qkv.dims[1], C = qkv.dims[2] / 3.0;
    double f = 10.0 * B * S * S * C;
    return n.attr_b("causal", true) ? f / 2 : f;
  }
  if (IsSource(op)) return 0.0;
  // elementwise-ish: a few flops per output element
  double e = 0;
  for (auto& t : n.outputs) e += (double)t.numel();
  (void)numel;
  return 4.0 * e;
}

}  // namespace tepdist
