"""Graph builder + reverse-mode autodiff: the client-side lowering of a model into planner IR.

This plays the role of the reference's patched TF client (SURVEY §2.F): it produces ONE graph holding the
forward pass, the backward pass and the optimizer update, stamps `op_group` / `backward` on every node
(F4/F7: a forward op and the gradient ops derived from it share a group id; optimizer slots and apply ops
take the variable's group) and records variables with their initialisers so the server can materialise
them shard-wise (F5 `init_from_remote`).
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence, Tuple

from ..ir import Graph, Node, TensorType, Value, numel


class GraphBuilder:
    def __init__(self, name: str = "step", compute_dtype: str = "bf16"):
        self.g = Graph(name)
        self.cd = compute_dtype
        self._scope: List[str] = []

    # ------------------------------------------------------------------ helpers
    def _n(self, op, inputs, outs, attrs=None, name="", group=None) -> Node:
        full = "/".join(self._scope + [name]) if name else ""
        grp = self.g.new_group() if group is None else group
        return self.g.add(op, inputs, outs, attrs, full, grp)

    def scope(self, name: str):
        b = self

        class _S:
            def __enter__(self_inner):
                b._scope.append(name)

            def __exit__(self_inner, *a):
                b._scope.pop()

        return _S()

    def t(self, v: Value) -> TensorType:
        return self.g.type_of(v)

    # ------------------------------------------------------------------ sources
    def parameter(self, name: str, shape: Sequence[int], init: Dict[str, Any], compute_dtype: Optional[str] = None,
                  decay: Optional[bool] = None) -> Value:
        """A trainable variable.  `init` is the RNG/constant spec the server uses to fill (its shard of) the
        variable: {"kind": "normal"|"uniform"|"truncated_normal"|"constant", "mean","std","lo","hi","value","seed"}."""
        cdt = compute_dtype or (self.cd if len(shape) >= 2 else "f32")
        full = "/".join(self._scope + [name])
        n = self.g.add("parameter", [], [TensorType(tuple(shape), cdt)],
                       {"init": init, "decay": bool(len(shape) >= 2 if decay is None else decay)}, full, self.g.new_group())
        return n.out()

    def input(self, name: str, shape: Sequence[int], dtype: str) -> Value:
        return self.g.add("input", [], [TensorType(tuple(shape), dtype)], {}, name, self.g.new_group()).out()

    def constant(self, value: float, shape: Sequence[int] = (), dtype: str = "f32") -> Value:
        return self._n("constant", [], [TensorType(tuple(shape), dtype)], {"value": value}).out()

    # ------------------------------------------------------------------ macro ops (map 1:1 onto sm_100a kernels)
    def embedding(self, tokens: Value, wte: Value, wpe: Value, name="embed") -> Value:
        B, S = self.t(tokens).shape
        C = self.t(wte).shape[1]
        return self._n("embedding", [tokens, wte, wpe], [TensorType((B, S, C), self.t(wte).dtype)], {}, name).out()

    def layernorm(self, x: Value, gamma: Value, beta: Value, eps: float = 1e-5, name="ln") -> Value:
        return self._n("layernorm", [x, gamma, beta], [self.t(x)], {"eps": eps}, name).out()

    def linear(self, x: Value, w: Value, b: Optional[Value] = None, residual: Optional[Value] = None,
               name="linear") -> Value:
        """y[..., N] = x[..., K] @ w[N, K]^T (+ b) (+ residual)."""
        xs, ws = self.t(x).shape, self.t(w).shape
        assert xs[-1] == ws[1], (xs, ws)
        ins = [x, w]
        attrs = {"bias": b is not None, "residual": residual is not None}
        if b is not None:
            ins.append(b)
        if residual is not None:
            ins.append(residual)
        return self._n("linear", ins, [TensorType(tuple(xs[:-1]) + (ws[0],), self.t(x).dtype)], attrs, name).out()

    def gelu(self, x: Value, name="gelu") -> Value:
        return self._n("gelu", [x], [self.t(x)], {}, name).out()

    def attention(self, qkv: Value, heads: int, causal: bool = True, segments: Optional[Value] = None, name="attn") -> Value:
        """Fused attention over qkv [B, S, 3C].  `segments` (int32 [B, S], optional): document ids; query i attends to key j
        only if segments[i] == segments[j] (and j <= i when causal)."""
        B, S, C3 = self.t(qkv).shape
        C = C3 // 3
        ins = [qkv]
        if segments is not None:
            assert tuple(self.t(segments).shape) == (B, S) and self.t(segments).dtype == "i32", self.t(segments)
            ins.append(segments)
        n = self._n("attention", ins, [TensorType((B, S, C), self.t(qkv).dtype), TensorType((B, heads, S), "f32")],
                    {"heads": heads, "causal": causal}, name)
        return n.out(0)

    def softmax_xent(self, logits: Value, labels: Value, vocab: Optional[int] = None, name="loss") -> Value:
        """Mean token cross-entropy.  Output 1 is d(loss)/d(logits), produced by the same fused kernel."""
        lt = self.t(logits)
        n = self._n("softmax_xent", [logits, labels], [TensorType((), "f32"), lt],
                    {"vocab": vocab or lt.shape[-1]}, name)
        return n.out(0)

    # ------------------------------------------------------------------ generic (HLO-like) ops
    def matmul(self, a: Value, b: Value, ta: bool = False, tb: bool = False, name="matmul") -> Value:
        """Batched dot: leading dims are batch dims (must match); contracts a's last (or -2 if ta) with b's -2 (or -1 if tb)."""
        sa, sb = list(self.t(a).shape), list(self.t(b).shape)
        m, ka = (sa[-1], sa[-2]) if ta else (sa[-2], sa[-1])
        kb, n = (sb[-1], sb[-2]) if tb else (sb[-2], sb[-1])
        assert ka == kb, (sa, sb, ta, tb)
        batch = sa[:-2] if len(sa) >= len(sb) else sb[:-2]
        return self._n("matmul", [a, b], [TensorType(tuple(batch) + (m, n), self.t(a).dtype)], {"ta": ta, "tb": tb}, name).out()

    def einsum(self, eq: str, a: Value, b: Value, name="einsum") -> Value:
        """Two-operand einsum kept as one planner 'dot' (batch / contracting / free dims come from the equation);
        this is how expert parallelism emerges (reference: examples/gpt_moe/layers/moe_layers.py:425-446)."""
        lhs, out = eq.replace(" ", "").split("->")
        ia, ib = lhs.split(",")
        dims: Dict[str, int] = {}
        for s, v in ((ia, a), (ib, b)):
            for ch, d in zip(s, self.t(v).shape):
                assert dims.setdefault(ch, d) == d, (eq, ch)
        return self._n("einsum", [a, b], [TensorType(tuple(dims[c] for c in out), self.t(a).dtype)], {"eq": eq}, name).out()

    def _ew(self, op: str, ins: Sequence[Value], name: str, attrs=None, dtype=None) -> Value:
        t0 = self.t(ins[0])
        shape = t0.shape
        for v in ins[1:]:
            s = self.t(v).shape
            if numel(s) > numel(shape):
                shape = s
        return self._n(op, list(ins), [TensorType(shape, dtype or t0.dtype)], attrs or {}, name).out()

    def add(self, x, y, name="add"): return self._ew("add", [x, y], name)
    def sub(self, x, y, name="sub"): return self._ew("sub", [x, y], name)
    def mul(self, x, y, name="mul"): return self._ew("mul", [x, y], name)
    def div(self, x, y, name="div"): return self._ew("div", [x, y], name)
    def relu(self, x, name="relu"): return self._ew("relu", [x], name)
    def tanh(self, x, name="tanh"): return self._ew("tanh", [x], name)
    def exp(self, x, name="exp"): return self._ew("exp", [x], name)
    def log(self, x, name="log"): return self._ew("log", [x], name)
    def neg(self, x, name="neg"): return self._ew("neg", [x], name)
    def scale(self, x, alpha: float, name="scale"): return self._ew("scale", [x], name, {"alpha": alpha})
    def cast(self, x, dtype: str, name="cast"): return self._ew("cast", [x], name, {"dtype": dtype}, dtype)

    # ---- further elementwise / structural ops (traced torch graphs bring them along; rules: csrc/rules.cc)
    def sqrt(self, x, name="sqrt"): return self._ew("sqrt", [x], name)
    def rsqrt(self, x, name="rsqrt"): return self._ew("rsqrt", [x], name)
    def sigmoid(self, x, name="sigmoid"): return self._ew("sigmoid", [x], name)
    def abs(self, x, name="abs"): return self._ew("abs", [x], name)
    def maximum(self, x, y, name="maximum"): return self._ew("maximum", [x, y], name)
    def minimum(self, x, y, name="minimum"): return self._ew("minimum", [x, y], name)
    def compare(self, x, y, direction: str = "gt", name="compare"): return self._ew("compare", [x, y], name, {"direction": direction}, "bool")

    def select(self, pred: Value, a: Value, b_: Value, name="select") -> Value:
        shape = max((self.t(v).shape for v in (pred, a, b_)), key=numel)
        return self._n("select", [pred, a, b_], [TensorType(shape, self.t(a).dtype)], {}, name).out()

    def reverse(self, x: Value, dims: Sequence[int], name="reverse") -> Value:
        return self._n("reverse", [x], [self.t(x)], {"dims": [d % len(self.t(x).shape) for d in dims]}, name).out()

    def sort(self, x: Value, axis: int = -1, descending: bool = False, name="sort") -> Value:
        return self._n("sort", [x], [self.t(x)], {"axis": axis % len(self.t(x).shape), "descending": descending}, name).out()

    def iota(self, shape: Sequence[int], dim: int, dtype: str = "i32", name="iota") -> Value:
        return self._n("iota", [], [TensorType(tuple(shape), dtype)], {"dim": dim}, name).out()

    def pad(self, x: Value, low: Sequence[int], high: Sequence[int], value: float = 0.0, name="pad") -> Value:
        s = self.t(x).shape
        out = tuple(d + lo + hi for d, lo, hi in zip(s, low, high))
        return self._n("pad", [x], [TensorType(out, self.t(x).dtype)], {"low": list(low), "high": list(high), "value": value}, name).out()

    def reduce_window(self, x: Value, window: Sequence[int], strides: Sequence[int], kind: str = "max", name="reduce_window") -> Value:
        """Unpadded window reduction over an N-d tensor (window / stride 1 on the dims it does not act along)."""
        s = self.t(x).shape
        out = tuple((d - w) // st + 1 for d, w, st in zip(s, window, strides))
        return self._n("reduce_window", [x], [TensorType(out, self.t(x).dtype)],
                       {"window": list(window), "strides": list(strides), "padding": [0] * (2 * len(s)), "kind": kind}, name).out()

    def softmax(self, x: Value, axis: int = -1, name="softmax") -> Value:
        return self._n("softmax", [x], [self.t(x)], {"axis": axis % len(self.t(x).shape)}, name).out()

    def reduce_sum(self, x: Value, axes: Sequence[int], keepdims=False, name="reduce_sum") -> Value:
        return self._reduce("reduce_sum", x, axes, keepdims, name)

    def reduce_mean(self, x: Value, axes: Sequence[int], keepdims=False, name="reduce_mean") -> Value:
        return self._reduce("reduce_mean", x, axes, keepdims, name)

    def reduce_max(self, x: Value, axes: Sequence[int], keepdims=False, name="reduce_max") -> Value:
        return self._reduce("reduce_max", x, axes, keepdims, name)

    def _reduce(self, op, x, axes, keepdims, name):
        s = self.t(x).shape
        axes = sorted(a % len(s) for a in axes)
        out = tuple((1 if i in axes else d) for i, d in enumerate(s)) if keepdims else tuple(d for i, d in enumerate(s) if i not in axes)
        return self._n(op, [x], [TensorType(out, self.t(x).dtype)], {"axes": axes, "keepdims": keepdims}, name).out()

    def reshape(self, x: Value, shape: Sequence[int], name="reshape") -> Value:
        shape = list(shape)
        if -1 in shape:
            i = shape.index(-1)
            shape[i] = numel(self.t(x).shape) // max(1, -numel(shape))
        assert numel(shape) == numel(self.t(x).shape), (shape, self.t(x).shape)
        return self._n("reshape", [x], [TensorType(tuple(shape), self.t(x).dtype)], {"shape": list(shape)}, name).out()

    def transpose(self, x: Value, perm: Sequence[int], name="transpose") -> Value:
        s = self.t(x).shape
        return self._n("transpose", [x], [TensorType(tuple(s[p] for p in perm), self.t(x).dtype)], {"perm": list(perm)}, name).out()

    def broadcast(self, x: Value, shape: Sequence[int], dims: Sequence[int], name="broadcast") -> Value:
        """HLO-style broadcast: operand dim i maps to output dim dims[i]."""
        return self._n("broadcast", [x], [TensorType(tuple(shape), self.t(x).dtype)], {"dims": list(dims), "shape": list(shape)}, name).out()

    def slice(self, x: Value, starts: Sequence[int], limits: Sequence[int], name="slice") -> Value:
        out = tuple(l - s for s, l in zip(starts, limits))
        return self._n("slice", [x], [TensorType(out, self.t(x).dtype)], {"starts": list(starts), "limits": list(limits)}, name).out()

    def concat(self, xs: Sequence[Value], axis: int, name="concat") -> Value:
        s = list(self.t(xs[0]).shape)
        s[axis] = sum(self.t(v).shape[axis] for v in xs)
        return self._n("concat", list(xs), [TensorType(tuple(s), self.t(xs[0]).dtype)], {"axis": axis}, name).out()

    def gather_rows(self, table: Value, idx: Value, name="gather") -> Value:
        """out[..., :] = table[idx[...], :] (embedding-style gather)."""
        return self._n("gather", [table, idx], [TensorType(self.t(idx).shape + self.t(table).shape[1:], self.t(table).dtype)], {}, name).out()

    def one_hot(self, idx: Value, depth: int, dtype: Optional[str] = None, name="one_hot") -> Value:
        return self._n("one_hot", [idx], [TensorType(self.t(idx).shape + (depth,), dtype or self.cd)], {"depth": depth}, name).out()

    def moe_dispatch_mask(self, gates: Value, capacity: int, top_k: int = 2, dtype: Optional[str] = None,
                          name="dispatch_mask") -> Value:
        """GShard-style top-k gating with per-expert capacity: gates [G,S,E] (probabilities) -> combine weights
        [G,S,E,C] (zero where a token is dropped).  (reference: examples/gpt_moe/layers/moe_layers.py top2 gating)"""
        G_, S_, E = self.t(gates).shape
        return self._n("moe_dispatch_mask", [gates], [TensorType((G_, S_, E, capacity), dtype or self.cd)],
                       {"capacity": capacity, "top_k": top_k}, name).out()

    # conv stack (Wide-ResNet): NCHW, weights OIHW; executed through cuDNN exactly as the reference does (K9)
    def conv2d(self, x: Value, w: Value, stride: int = 1, padding: int = 0, name="conv") -> Value:
        N, C, H, W = self.t(x).shape
        O, I, kh, kw = self.t(w).shape
        assert I == C
        Ho = (H + 2 * padding - kh) // stride + 1
        Wo = (W + 2 * padding - kw) // stride + 1
        return self._n("conv2d", [x, w], [TensorType((N, O, Ho, Wo), self.t(x).dtype)], {"stride": stride, "padding": padding}, name).out()

    def batchnorm(self, x: Value, gamma: Value, beta: Value, eps=1e-5, name="bn") -> Value:
        """Training-mode batch norm over (N,H,W) (batch statistics)."""
        return self._n("batchnorm", [x, gamma, beta], [self.t(x)], {"eps": eps}, name).out()

    def maxpool2d(self, x: Value, k: int, stride: int, padding: int = 0, name="maxpool") -> Value:
        N, C, H, W = self.t(x).shape
        Ho = (H + 2 * padding - k) // stride + 1
        Wo = (W + 2 * padding - k) // stride + 1
        return self._n("maxpool2d", [x], [TensorType((N, C, Ho, Wo), self.t(x).dtype)], {"k": k, "stride": stride, "padding": padding}, name).out()

    def global_avgpool(self, x: Value, name="gap") -> Value:
        N, C, H, W = self.t(x).shape
        return self._n("global_avgpool", [x], [TensorType((N, C), self.t(x).dtype)], {}, name).out()

    # user sharding annotations (xla_sharding.split / replicate equivalents, SURVEY Appendix F)
    def annotate_split(self, v: Value, dim: int, num: int) -> Value:
        self.g.nodes[v.node].attrs.setdefault("sharding", {})[str(v.idx)] = {"dim": dim, "num": num}
        return v

    def annotate_replicate(self, v: Value) -> Value:
        self.g.nodes[v.node].attrs.setdefault("sharding", {})[str(v.idx)] = {"dim": -1, "num": 1}
        return v


# ====================================================================================== autodiff
def _sum_grads(b: GraphBuilder, gs: List[Value], group: int) -> Value:
    acc = gs[0]
    for g in gs[1:]:
        n = b.g.add("add", [acc, g], [b.t(acc)], {}, "", group, True)
        acc = n.out()
    return acc


def _unbroadcast(b: GraphBuilder, g: Value, target_shape, group) -> Value:
    gs = b.t(g).shape
    if tuple(gs) == tuple(target_shape):
        return g
    # sum leading / size-1 dims
    lead = len(gs) - len(target_shape)
    axes = list(range(lead)) + [lead + i for i, d in enumerate(target_shape) if d == 1 and gs[lead + i] != 1]
    out_shape = tuple(d for i, d in enumerate(gs) if i not in axes)
    n = b.g.add("reduce_sum", [g], [TensorType(out_shape, b.t(g).dtype)], {"axes": axes, "keepdims": False}, "", group, True)
    v = n.out()
    if out_shape != tuple(target_shape):
        v = b.g.add("reshape", [v], [TensorType(tuple(target_shape), b.t(g).dtype)], {"shape": list(target_shape)}, "", group, True).out()
    return v


def backward(b: GraphBuilder, loss: Value) -> Dict[int, Value]:
    """Appends the backward pass for scalar `loss`; returns {parameter node id -> gradient value (fp32)}."""
    g = b.g
    grads: Dict[Tuple[int, int], List[Value]] = {}
    n_fwd = len(g.nodes)
    # which nodes need grad (reach a parameter)
    needs = [False] * n_fwd
    for n in g.nodes[:n_fwd]:
        if n.op == "parameter":
            needs[n.id] = True
        elif n.op not in ("input", "constant", "state"):
            needs[n.id] = any(needs[v.node] for v in n.inputs)
    one = g.add("constant", [], [TensorType((), "f32")], {"value": 1.0}, "dloss", g.nodes[loss.node].group, True).out()
    grads[loss.key()] = [one]

    def B(op, ins, outs, attrs, grp):
        return g.add(op, ins, outs, attrs, "", grp, True)

    def push(v: Value, gv: Value):
        if needs[v.node]:
            grads.setdefault(v.key(), []).append(gv)

    for n in reversed(g.nodes[:n_fwd]):
        if not needs[n.id] or n.op == "parameter":
            continue
        outs_g = [(_sum_grads(b, grads[(n.id, i)], n.group) if (n.id, i) in grads else None) for i in range(len(n.outputs))]
        if all(x is None for x in outs_g):
            continue
        dy = outs_g[0]
        grp = n.group
        T = g.type_of
        if n.op == "softmax_xent":
            logits = n.inputs[0]
            dl = Value(n.id, 1)  # already d loss / d logits for dloss = 1 (root); general case scales it
            if grads[(n.id, 0)] != [one]:
                dl = B("mul", [dl, dy], [T(dl)], {}, grp).out()
            push(logits, dl)
        elif n.op == "linear":
            x, w = n.inputs[0], n.inputs[1]
            k = 2
            if needs[x.node]:
                push(x, B("linear_dgrad", [dy, w], [T(x)], {}, grp).out())
            push(w, B("linear_wgrad", [dy, x], [TensorType(T(w).shape, "f32")], {}, grp).out())
            if n.attrs.get("bias"):
                bv = n.inputs[k]; k += 1
                push(bv, B("colsum", [dy], [TensorType(T(bv).shape, "f32")], {}, grp).out())
            if n.attrs.get("residual"):
                push(n.inputs[k], dy)
        elif n.op == "layernorm":
            x, gm, bt = n.inputs
            nb = B("layernorm_bwd", [dy, x, gm], [T(x), TensorType(T(gm).shape, "f32"), TensorType(T(bt).shape, "f32")],
                   {"eps": n.attrs["eps"]}, grp)
            push(x, nb.out(0)); push(gm, nb.out(1)); push(bt, nb.out(2))
        elif n.op == "gelu":
            push(n.inputs[0], B("gelu_bwd", [dy, n.inputs[0]], [T(n.inputs[0])], {}, grp).out())
        elif n.op == "attention":
            qkv = n.inputs[0]
            push(qkv, B("attention_bwd", [dy, qkv, Value(n.id, 0), Value(n.id, 1)] + list(n.inputs[1:]), [T(qkv)], dict(n.attrs),
                        grp).out())
        elif n.op == "embedding":
            tok, wte, wpe = n.inputs
            nb = B("embedding_bwd", [tok, dy], [TensorType(T(wte).shape, "f32"), TensorType(T(wpe).shape, "f32")], {}, grp)
            push(wte, nb.out(0)); push(wpe, nb.out(1))
        elif n.op in ("add", "sub"):
            x, y = n.inputs
            push(x, _unbroadcast(b, dy, T(x).shape, grp))
            gy = dy if n.op == "add" else B("neg", [dy], [T(dy)], {}, grp).out()
            push(y, _unbroadcast(b, gy, T(y).shape, grp))
        elif n.op == "mul":
            x, y = n.inputs
            push(x, _unbroadcast(b, B("mul", [dy, y], [T(dy)], {}, grp).out(), T(x).shape, grp))
            push(y, _unbroadcast(b, B("mul", [dy, x], [T(dy)], {}, grp).out(), T(y).shape, grp))
        elif n.op == "div":
            x, y = n.inputs
            gx = B("div", [dy, y], [T(dy)], {}, grp).out()
            push(x, _unbroadcast(b, gx, T(x).shape, grp))
            if needs[y.node]:
                t1 = B("mul", [gx, Value(n.id, 0)], [T(dy)], {}, grp).out()
                push(y, _unbroadcast(b, B("neg", [t1], [T(dy)], {}, grp).out(), T(y).shape, grp))
        elif n.op == "scale":
            push(n.inputs[0], B("scale", [dy], [T(dy)], {"alpha": n.attrs["alpha"]}, grp).out())
        elif n.op == "neg":
            push(n.inputs[0], B("neg", [dy], [T(dy)], {}, grp).out())
        elif n.op == "cast":
            push(n.inputs[0], B("cast", [dy], [T(n.inputs[0])], {"dtype": T(n.inputs[0]).dtype}, grp).out())
        elif n.op == "relu":
            push(n.inputs[0], B("relu_bwd", [dy, Value(n.id, 0)], [T(dy)], {}, grp).out())
        elif n.op == "tanh":
            push(n.inputs[0], B("tanh_bwd", [dy, Value(n.id, 0)], [T(dy)], {}, grp).out())
        elif n.op == "exp":
            push(n.inputs[0], B("mul", [dy, Value(n.id, 0)], [T(dy)], {}, grp).out())
        elif n.op == "log":
            push(n.inputs[0], B("div", [dy, n.inputs[0]], [T(dy)], {}, grp).out())
        elif n.op == "softmax":
            push(n.inputs[0], B("softmax_bwd", [dy, Value(n.id, 0)], [T(dy)], {"axis": n.attrs["axis"]}, grp).out())
        elif n.op in ("reduce_sum", "reduce_mean"):
            x = n.inputs[0]
            xs = T(x).shape
            axes = n.attrs["axes"]
            gy = dy
            if n.op == "reduce_mean":
                cnt = 1
                for a in axes:
                    cnt *= xs[a]
                gy = B("scale", [gy], [T(gy)], {"alpha": 1.0 / cnt}, grp).out()
            kept = [i for i in range(len(xs)) if i not in axes]
            if n.attrs.get("keepdims"):
                kshape = tuple(d for i, d in enumerate(xs) if i not in axes)
                gy = B("reshape", [gy], [TensorType(kshape, T(gy).dtype)], {"shape": list(kshape)}, grp).out()
            push(x, B("broadcast", [gy], [TensorType(xs, T(gy).dtype)], {"dims": kept, "shape": list(xs)}, grp).out())
        elif n.op == "reshape":
            x = n.inputs[0]
            push(x, B("reshape", [dy], [TensorType(T(x).shape, T(dy).dtype)], {"shape": list(T(x).shape)}, grp).out())
        elif n.op == "transpose":
            perm = n.attrs["perm"]
            inv = [perm.index(i) for i in range(len(perm))]
            push(n.inputs[0], B("transpose", [dy], [TensorType(T(n.inputs[0]).shape, T(dy).dtype)], {"perm": inv}, grp).out())
        elif n.op == "broadcast":
            x = n.inputs[0]
            dims = n.attrs["dims"]
            axes = [i for i in range(len(T(dy).shape)) if i not in dims]
            push(x, B("reduce_sum", [dy], [TensorType(T(x).shape, T(dy).dtype)], {"axes": axes, "keepdims": False}, grp).out())
        elif n.op == "matmul":
            a, bb = n.inputs
            ta, tb = n.attrs["ta"], n.attrs["tb"]
            # dA = dY B^T (or B dY^T when ta), dB = A^T dY (or dY^T A when tb)
            if needs[a.node]:
                if not ta:
                    ga = B("matmul", [dy, bb], [T(a)], {"ta": False, "tb": not tb}, grp).out()
                else:
                    ga = B("matmul", [bb, dy], [T(a)], {"ta": tb, "tb": True}, grp).out()
                push(a, _unbroadcast(b, ga, T(a).shape, grp))
            if needs[bb.node]:
                if not tb:
                    gb = B("matmul", [a, dy], [TensorType(T(dy).shape[:-2] + T(bb).shape[-2:], T(bb).dtype)], {"ta": not ta, "tb": False}, grp).out()
                else:
                    gb = B("matmul", [dy, a], [TensorType(T(dy).shape[:-2] + T(bb).shape[-2:], T(bb).dtype)], {"ta": True, "tb": ta}, grp).out()
                push(bb, _unbroadcast(b, gb, T(bb).shape, grp))
        elif n.op == "einsum":
            a, bb = n.inputs
            lhs, out = n.attrs["eq"].replace(" ", "").split("->")
            ia, ib = lhs.split(",")
            if needs[a.node]:
                push(a, B("einsum", [dy, bb], [T(a)], {"eq": f"{out},{ib}->{ia}"}, grp).out())
            if needs[bb.node]:
                push(bb, B("einsum", [a, dy], [T(bb)], {"eq": f"{ia},{out}->{ib}"}, grp).out())
        elif n.op == "gather":
            table, idx = n.inputs
            push(table, B("scatter_add", [idx, dy], [TensorType(T(table).shape, "f32")], {}, grp).out())
        elif n.op == "slice":
            x = n.inputs[0]
            push(x, B("pad_zero", [dy], [TensorType(T(x).shape, T(dy).dtype)], {"starts": n.attrs["starts"], "shape": list(T(x).shape)}, grp).out())
        elif n.op == "concat":
            off = 0
            ax = n.attrs["axis"]
            for v in n.inputs:
                s = T(v).shape
                st = [0] * len(s); lm = list(T(dy).shape)
                st[ax] = off; lm[ax] = off + s[ax]
                push(v, B("slice", [dy], [TensorType(s, T(dy).dtype)], {"starts": st, "limits": lm}, grp).out())
                off += s[ax]
        elif n.op == "conv2d":
            x, w = n.inputs
            if needs[x.node]:
                push(x, B("conv2d_dgrad", [dy, w], [T(x)], dict(n.attrs), grp).out())
            push(w, B("conv2d_wgrad", [dy, x], [TensorType(T(w).shape, "f32")], dict(n.attrs), grp).out())
        elif n.op == "batchnorm":
            x, gm, bt = n.inputs
            nb = B("batchnorm_bwd", [dy, x, gm], [T(x), TensorType(T(gm).shape, "f32"), TensorType(T(bt).shape, "f32")], dict(n.attrs), grp)
            push(x, nb.out(0)); push(gm, nb.out(1)); push(bt, nb.out(2))
        elif n.op == "maxpool2d":
            push(n.inputs[0], B("maxpool2d_bwd", [dy, n.inputs[0], Value(n.id, 0)], [T(n.inputs[0])], dict(n.attrs), grp).out())
        elif n.op == "global_avgpool":
            push(n.inputs[0], B("global_avgpool_bwd", [dy], [T(n.inputs[0])], {}, grp).out())
        elif n.op == "moe_dispatch_mask":
            gts = n.inputs[0]
            push(gts, B("moe_dispatch_mask_bwd", [dy, gts], [T(gts)], dict(n.attrs), grp).out())
        elif n.op == "sqrt":       # d sqrt(x) = dy / (2 y)
            half = B("scale", [dy], [T(dy)], {"alpha": 0.5}, grp).out()
            push(n.inputs[0], B("div", [half, Value(n.id, 0)], [T(dy)], {}, grp).out())
        elif n.op == "rsqrt":      # d x^-1/2 = -1/2 y^3 dy
            y2 = B("mul", [Value(n.id, 0), Value(n.id, 0)], [T(dy)], {}, grp).out()
            y3 = B("mul", [y2, Value(n.id, 0)], [T(dy)], {}, grp).out()
            push(n.inputs[0], B("scale", [B("mul", [dy, y3], [T(dy)], {}, grp).out()], [T(dy)], {"alpha": -0.5}, grp).out())
        elif n.op == "sigmoid":
            push(n.inputs[0], B("sigmoid_bwd", [dy, Value(n.id, 0)], [T(dy)], {}, grp).out())
        elif n.op == "abs":
            push(n.inputs[0], B("mul", [dy, B("sign", [n.inputs[0]], [T(dy)], {}, grp).out()], [T(dy)], {}, grp).out())
        elif n.op in ("maximum", "minimum"):
            x, y = n.inputs
            take_x = B("compare", [x, y], [TensorType(T(dy).shape, "bool")], {"direction": "ge" if n.op == "maximum" else "le"}, grp).out()
            zero = B("constant", [], [TensorType((), T(dy).dtype)], {"value": 0.0}, grp).out()
            push(x, _unbroadcast(b, B("select", [take_x, dy, zero], [T(dy)], {}, grp).out(), T(x).shape, grp))
            push(y, _unbroadcast(b, B("select", [take_x, zero, dy], [T(dy)], {}, grp).out(), T(y).shape, grp))
        elif n.op == "select":
            pred, x, y = n.inputs
            zero = B("constant", [], [TensorType((), T(dy).dtype)], {"value": 0.0}, grp).out()
            push(x, _unbroadcast(b, B("select", [pred, dy, zero], [T(dy)], {}, grp).out(), T(x).shape, grp))
            push(y, _unbroadcast(b, B("select", [pred, zero, dy], [T(dy)], {}, grp).out(), T(y).shape, grp))
        elif n.op == "reverse":
            push(n.inputs[0], B("reverse", [dy], [T(dy)], {"dims": n.attrs["dims"]}, grp).out())
        elif n.op == "pad":
            x = n.inputs[0]
            lo = n.attrs["low"]
            lim = [l + d for l, d in zip(lo, T(x).shape)]
            push(x, B("slice", [dy], [TensorType(T(x).shape, T(dy).dtype)], {"starts": list(lo), "limits": lim}, grp).out())
        elif n.op == "reduce_window":
            x = n.inputs[0]
            push(x, B("select_and_scatter", [x, dy], [T(x)], dict(n.attrs), grp).out())
        elif n.op in ("one_hot", "reduce_max", "compare", "iota", "sort", "sign"):
            pass
        else:
            raise NotImplementedError(f"no vjp for op '{n.op}'")

    out: Dict[int, Value] = {}
    for pn in g.params():
        key = (pn.id, 0)
        if key in grads:
            gv = _sum_grads(b, grads[key], pn.group)
            if g.type_of(gv).dtype != "f32":
                gv = g.add("cast", [gv], [TensorType(g.type_of(gv).shape, "f32")], {"dtype": "f32"}, "", pn.group, True).out()
            out[pn.id] = gv
    return out


OPTIMIZERS = ("sgd", "momentum", "adam", "adamw", "lamb", "adafactor", "sm3")


def apply_optimizer(b: GraphBuilder, grads: Dict[int, Value], kind: str = "adamw", **hp) -> None:
    """Appends one apply node per variable (+ its slot `state` nodes) and registers in/out aliases.

    Optimizers of the reference's example suites (examples/GPT2/optimizers.py, examples/gpt_moe/optimizers/*):
      sgd        p -= lr g
      momentum   v = mu v + g; p -= lr v                                        (hp: lr, momentum)
      adam       AdamW with weight_decay = 0
      adamw      decoupled weight decay on variables with decay=True            (hp: lr, beta1, beta2, eps, weight_decay)
      lamb       Adam direction (+ wd p), scaled per variable by |p| / |update| (lamb_weight_decay_optimizer.py:121-154)
      adafactor  factored second moments for rank >= 2 (row / column means), update clipping by RMS, step scaled by
                 RMS(p); decay rate 1 - t^-0.8                                   (adafactor.py:127-139 defaults)
      sm3        one accumulator per dimension, nu = min_i acc_i + g^2, acc_i = max over the other dims (sm3.py:92-165)
    Slots of the non-elementwise optimizers have reduced shapes; the planner's rules (rules.cc AdafactorRule / Sm3Rule) lay
    them out consistently with the variable and the executor completes their reductions across shards."""
    g = b.g
    if kind not in OPTIMIZERS:
        raise ValueError(f"optimizer '{kind}': expected one of {OPTIMIZERS}")
    if kind == "adam":
        kind, hp = "adamw", {**hp, "weight_decay": 0.0}
    g.meta["optimizer"] = {"kind": kind, **hp}
    zeros = {"kind": "constant", "value": 0.0}

    def slot(pn, suffix, shape):
        return g.add("state", [], [TensorType(tuple(shape), "f32")], {"init": zeros, "slot_of": pn.id}, pn.name + suffix, pn.group)

    def finish(pn, op, slots, attrs):
        n = g.add(op, [pn.out(), gv] + [s_.out() for s_ in slots], [TensorType(pn.outputs[0].shape, pn.outputs[0].dtype)] +
                  [TensorType(s_.outputs[0].shape, "f32") for s_ in slots], attrs, pn.name + "/apply", pn.group, True)
        g.updates[pn.id] = n.out(0)
        for i, s_ in enumerate(slots):
            g.updates[s_.id] = n.out(i + 1)

    for pid, gv in grads.items():
        pn = g.nodes[pid]
        shape = tuple(pn.outputs[0].shape)
        decay = pn.attrs.get("decay", True)
        if kind == "sgd":
            finish(pn, "apply_sgd", [], dict(hp))
        elif kind == "momentum":
            finish(pn, "apply_momentum", [slot(pn, "/mom", shape)], dict(hp))
        elif kind == "adamw":
            finish(pn, "apply_adamw", [slot(pn, "/m", shape), slot(pn, "/v", shape)], {**hp, "decay": decay})
        elif kind == "lamb":
            finish(pn, "apply_lamb", [slot(pn, "/m", shape), slot(pn, "/v", shape)], {**hp, "decay": decay})
        elif kind == "adafactor":
            if len(shape) >= 2 and hp.get("factored", True):
                slots = [slot(pn, "/vr", shape[:-1]), slot(pn, "/vc", shape[:-2] + shape[-1:])]
            else:
                slots = [slot(pn, "/vf", shape)]
            finish(pn, "apply_adafactor", slots, {**hp, "decay": decay})
        elif kind == "sm3":
            slots = [slot(pn, f"/acc{i}", (d,)) for i, d in enumerate(shape)] if len(shape) > 1 else [slot(pn, "/acc", shape)]
            if hp.get("momentum", 0.0) > 0:
                slots.append(slot(pn, "/mom", shape))
            finish(pn, "apply_sm3", slots, dict(hp))


def build_training_step(b: GraphBuilder, loss: Value, optimizer: str = "adamw", **hp) -> Graph:
    grads = backward(b, loss)
    apply_optimizer(b, grads, optimizer, **hp)
    b.g.outputs = [loss]
    b.g.validate()
    return b.g
