"""Graph executor: runs one (sub-)graph of planner IR on one device.

Design (B200-first, replaces XLA executables + thunk sequences of the reference — SURVEY §3.3/3.4):
  * variables live on the device across steps in FLAT buffers (fp32 master, bf16 compute copy, fp32
    gradient accumulators, optimizer slots) so the optimizer update, gradient zeroing ("GAInit") and
    the data-parallel gradient reduction are each ONE kernel / collective over contiguous memory;
  * every node maps onto a hand-written sm_100a kernel (tepdist_b200.ops) on the hot path;
  * activations are freed by a liveness plan computed once (the reference's
    OutputBuffersLifeTimeTracker / MakeTaskGraphGCPlan, SURVEY D5/D6);
  * the whole step is captured into a CUDA graph after warm-up, so the host-side interpreter cost
    (the reference's per-thunk host loop) disappears from the steady state.
In-place update semantics (input/output aliasing of variables, Appendix E) are honoured by updating
the flat buffers directly.
"""
from __future__ import annotations

import os
from typing import Any, Callable, Dict, List, Optional, Tuple

import torch

from .. import ops
from ..ir import COLLECTIVE_OPS, SOURCE_OPS, Graph, Node, Value
from ..utils.init import init_tensor

# tensor-parallel plans: run `linear -> all_reduce [-> + bias] [-> + residual]` as GEMM -> all-reduce over peer memory
# (parallel/symm.py GemmAllReduceMC: GEMM into a multicast-bound buffer + ONE multimem reduction kernel with bias / residual
# fused) instead of GEMM + NCCL + separate adds.  Default in comm = "fused" mode (validated on 2 / 4 / 8 B200: 1.10x / 1.25x /
# 1.51x the NCCL arm of the same plan, profiles/round2); TEPDIST_TP_FUSED=0 or comm = "nccl" selects the library collectives.
TP_FUSED = os.environ.get("TEPDIST_TP_FUSED", "1") == "1"
# test hook: a factory (M, N, group, barrier) -> object with new_output() / __call__(x, w, out, bias, residual, b_mn) that
# stands in for parallel.symm.GemmAllReduce, so the executor-side chain fusion can be exercised on CPU (gloo) where the
# peer-memory kernels cannot run
TP_FUSED_IMPL = None
# GPT-MoE: dispatch / combine einsums whose mask comes from moe_dispatch_mask run as route-table row gathers (ops.moe_*), not as
# dense [G,S,E*C] x [G,S,M] GEMMs; TEPDIST_MOE_SPARSE=0 keeps the dense einsums (the comparator)
MOE_SPARSE = os.environ.get("TEPDIST_MOE_SPARSE", "1") == "1"
# weight gradients with a single producer are written with plain stores instead of fp32 atomics into a zero-filled slot
WGRAD_PLAIN_STORE = os.environ.get("TEPDIST_WGRAD_STORE", "1") == "1"

_TORCH_DTYPE = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32, "i32": torch.int32,
                "i64": torch.int64, "bool": torch.bool}
_ALIGN = 128  # elements; keeps every variable slice 16-B aligned in every dtype
FLAT_APPLY = ("apply_adamw", "apply_sgd")   # elementwise updates: may run over the flat buffers / fused sharded-optimizer kernels


def torch_dtype(name: str, device: torch.device) -> torch.dtype:
    if device.type == "cpu" and name in ("bf16", "f16"):
        return torch.float32  # CPU plumbing / oracle path computes in fp32
    return _TORCH_DTYPE[name]


def shard_of(t: torch.Tensor, attrs: Dict[str, Any], coords: Dict[int, int]) -> torch.Tensor:
    """Slice a full tensor down to this rank's shard following the shard_dims/nums/levels a transform recorded."""
    dims, nums, lvls = attrs.get("shard_dims", []), attrs.get("shard_nums", []), attrs.get("shard_levels", [])
    for d, n, l in zip(dims, nums, lvls):
        sz = t.shape[d] // n
        t = t.narrow(d, coords.get(int(l), 0) * sz, sz)
    return t


class VariableStore:
    """Flat device-resident storage for all variables of a graph (+ grads and optimizer slots)."""

    def __init__(self, graph: Graph, device: torch.device, seed: int = 0, coords: Optional[Dict[int, int]] = None,
                 tail: Optional[set] = None):
        self.device = device
        self.coords = coords or {}
        tail = tail or set()
        params = graph.params()
        # decayed variables first so the fused AdamW kernel can use a prefix length; variables whose optimizer
        # pattern is irregular (`tail`) go last so the flat sharded-optimizer range stays contiguous
        params = sorted(params, key=lambda n: (n.id in tail, not n.attrs.get("decay", True), n.id))
        self.regular_end = 0
        self.order = [n.id for n in params]
        self.offset: Dict[int, int] = {}
        self.shape: Dict[int, Tuple[int, ...]] = {}
        self.cdtype: Dict[int, str] = {}
        off = 0
        self.n_decay = 0
        for n in params:
            self.offset[n.id] = off
            self.shape[n.id] = tuple(n.outputs[0].shape)
            self.cdtype[n.id] = n.outputs[0].dtype
            sz = n.outputs[0].numel()
            off += (sz + _ALIGN - 1) // _ALIGN * _ALIGN
            if n.attrs.get("decay", True) and n.id not in tail:
                self.n_decay = off
            if n.id not in tail:
                self.regular_end = off
        self.total = max(off, _ALIGN)
        f32 = dict(dtype=torch.float32, device=device)
        self.master = torch.zeros(self.total, **f32)
        self.grad = torch.zeros(self.total, **f32)
        self.m: Optional[torch.Tensor] = None
        self.v: Optional[torch.Tensor] = None
        # variables whose first / second moments the EXECUTION keeps in the flat m / v buffers (set by the executor once it
        # knows its update scheme; None = every variable, the single-process fused update).  The sharded-optimizer path keeps
        # them there even though the plan's slot nodes are chunk-shaped -- those slot tensors are then never touched.
        self.flat_moment_pids: Optional[set] = None
        self.compute = (torch.zeros(self.total, dtype=torch.bfloat16, device=device)
                        if device.type == "cuda" else None)
        self.names = {n.id: n.name for n in params}
        # optimizer slots (`state` nodes): views into the flat m / v buffers when they have their variable's shape
        # (fused update path), separate tensors otherwise (e.g. ZeRO-sharded slots of a replicated variable)
        self.state: Dict[int, torch.Tensor] = {}
        self._state_nodes = [n for n in graph.nodes if n.op == "state"]
        for n in params:
            full = tuple(n.attrs.get("full_shape", self.shape[n.id]))
            # only this rank's shard is generated (bit-identical to slicing a fill of the full tensor, see utils/init.py)
            t = init_tensor(n.attrs.get("init", {"kind": "constant", "value": 0.0}), full, seed, n.name, shard=(n.attrs, self.coords))
            self.master_view(n.id).copy_(t.reshape(self.shape[n.id]).to(device))
        self.sync_compute()

    def grow(self, total: int) -> None:
        """Pad the flat buffers (bucket/chunk alignment for the sharded optimizer)."""
        def pad(t):
            if t is None:
                return None
            out = torch.zeros(total, dtype=t.dtype, device=t.device)
            out[:t.numel()].copy_(t)
            return out
        self.master, self.grad, self.m, self.v, self.compute = (pad(x) for x in (self.master, self.grad, self.m, self.v, self.compute))
        self.total = total
        self.state.clear()

    def make_symmetric(self, group) -> None:
        """Move the gradient and bf16 parameter buffers into peer-mapped memory (fused NVLink kernels)."""
        from ..parallel.symm import SymmetricBuffer
        gb = SymmetricBuffer(self.total * 4, group)
        pb = SymmetricBuffer(self.total * 2, group)
        g = gb.tensor(torch.float32, self.total)
        c = pb.tensor(torch.bfloat16, self.total)
        g.copy_(self.grad)
        c.copy_(self.compute)
        self.grad, self.compute = g, c
        self.symm_grad, self.symm_param = gb, pb
        # bf16 gradient wire (TEPDIST_GRAD_WIRE=bf16, the reference's FP16_COMM idea on the NVLS path): a bf16 staging copy of the
        # gradient buffer that the switch reduces with fp32 accumulation; half the NVLink bytes of the fp32 wire
        self.symm_grad16 = None
        if os.environ.get("TEPDIST_GRAD_WIRE", "f32") == "bf16" and gb.mc_ptr is not None:
            self.symm_grad16 = SymmetricBuffer(self.total * 2, group)

    def _flat_slot(self, n) -> bool:
        """First / second moment slots with their variable's shape live in the flat m / v buffers."""
        pid = n.attrs.get("slot_of")
        return (pid in self.shape and self.shape[pid] == tuple(n.outputs[0].shape)
                and (n.name.endswith("/m") or n.name.endswith("/v")))

    def moments_flat(self, pid: int) -> bool:
        return self.m is not None and (self.flat_moment_pids is None or pid in self.flat_moment_pids)

    def slot_is_live(self, n) -> bool:
        """A slot tensor outside the flat buffers that the execution really updates (not shadowed by flat moments)."""
        if n.id not in self.state or self._flat_slot(n):
            return False
        pid = n.attrs.get("slot_of")
        return not (self.moments_flat(pid) and (n.name.endswith("/m") or n.name.endswith("/v")))

    def ensure_slots(self, flat_moments: bool = False) -> None:
        """`flat_moments`: the graph updates with AdamW, whose flat paths (fused whole-buffer update, sharded-optimizer
        chunks) address m / v by FLAT offset even when every slot node of the plan is chunk-shaped -- always allocate them."""
        if self.m is None and (flat_moments or any(self._flat_slot(n) for n in self._state_nodes)):
            self.m = torch.zeros_like(self.master)
            self.v = torch.zeros_like(self.master)
        for n in self._state_nodes:
            if n.id in self.state:
                continue
            if self._flat_slot(n):
                buf = self.m if n.name.endswith("/m") else self.v
                self.state[n.id] = self._view(buf, n.attrs.get("slot_of"))
            else:   # sharded slots of a replicated variable, reduced-shape slots (Adafactor, SM3), momentum
                self.state[n.id] = torch.zeros(tuple(n.outputs[0].shape), dtype=torch.float32, device=self.device)

    def _view(self, buf: torch.Tensor, pid: int) -> torch.Tensor:
        o = self.offset[pid]
        n = 1
        for d in self.shape[pid]:
            n *= d
        return buf[o:o + n].view(self.shape[pid])

    def master_view(self, pid: int) -> torch.Tensor:
        return self._view(self.master, pid)

    def grad_view(self, pid: int) -> torch.Tensor:
        return self._view(self.grad, pid)

    def compute_view(self, pid: int) -> torch.Tensor:
        if self.compute is not None and self.cdtype[pid] == "bf16":
            return self._view(self.compute, pid)
        return self.master_view(pid)

    def sync_compute(self) -> None:
        if self.compute is not None:
            ops.cast_f32_bf16(self.master, self.compute)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        out = {self.names[p]: self.master_view(p).detach().clone() for p in self.order}
        if self.m is not None:
            out.update({self.names[p] + "/m": self._view(self.m, p).detach().clone() for p in self.order if self.moments_flat(p)})
            out.update({self.names[p] + "/v": self._view(self.v, p).detach().clone() for p in self.order if self.moments_flat(p)})
        for n in self._state_nodes:     # slots outside the flat buffers
            if self.slot_is_live(n):
                out[n.name] = self.state[n.id].detach().clone()
        return out

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for p in self.order:
            nm = self.names[p]
            if nm in sd:
                self.master_view(p).copy_(sd[nm].to(self.device))
            if nm + "/m" in sd and tuple(sd[nm + "/m"].shape) == self.shape[p]:     # (else: a separately sharded slot, below)
                self.ensure_slots(flat_moments=True)
                self._view(self.m, p).copy_(sd[nm + "/m"].to(self.device))
                self._view(self.v, p).copy_(sd[nm + "/v"].to(self.device))
        for n in self._state_nodes:
            if n.name in sd and not self._flat_slot(n) and tuple(sd[n.name].shape) == tuple(n.outputs[0].shape):
                self.ensure_slots()
                self.state[n.id].copy_(sd[n.name].to(self.device).reshape(self.state[n.id].shape))
        self.sync_compute()


class Executor:
    """Interprets a Graph on one device.  `grad_sync(flat_grad)` (optional) is called once between the
    backward and the optimizer nodes — the data-parallel hook (see parallel/dp.py)."""

    def __init__(self, graph: Graph, device: Optional[torch.device] = None, seed: int = 0,
                 grad_sync: Optional[Callable[[torch.Tensor], None]] = None, use_cuda_graph: bool = False,
                 collective: Optional[Any] = None, store: Optional[VariableStore] = None,
                 coords: Optional[Dict[int, int]] = None, comm_mode: str = "nccl"):
        self.g = graph
        self.device = device or torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self.coords = coords or {}
        self.comm_mode = comm_mode
        self._fz_static = self._analyze_flat_zero(graph) if collective is not None else None
        tail = self._fz_static["irregular_params"] if self._fz_static else set()
        self.store = store or VariableStore(graph, self.device, seed, self.coords, tail=tail)
        self.grad_sync = grad_sync
        self.collective = collective
        # timing-only mode (bench.py's exposed-communication measurement): every collective is replaced by a local
        # stand-in of the same output shape, the sharded optimizer touches only local memory.  Numerics are meaningless.
        self.dry_comm = os.environ.get("TEPDIST_DRY_COMM") == "1"
        if self.dry_comm and collective is not None:
            collective.dry = True
        self.step_count = 0
        self._tag = 0   # micro-batch tag for per-micro-batch side tables (pipeline interleaves micro-batches)
        self.use_cuda_graph = use_cuda_graph and self.device.type == "cuda"
        if self.use_cuda_graph and any(n.attrs.get("cp_levels") for n in graph.nodes) and os.environ.get("TEPDIST_CP_GRAPH") != "1":
            self.use_cuda_graph = False    # ring attention posts point-to-point batches per block: run the step eagerly
        self._rings: Dict[Tuple[int, ...], Any] = {}
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._static_in: Dict[str, torch.Tensor] = {}
        self._static_out: List[torch.Tensor] = []
        from .optimizers import HYPER_SIZE    # (the CUDA kernels read the first four entries)
        self.hyper = torch.zeros(HYPER_SIZE, dtype=torch.float32, device=self.device)
        self._hyper_host = (torch.zeros(HYPER_SIZE, dtype=torch.float32).pin_memory() if self.device.type == "cuda"
                            else torch.zeros(HYPER_SIZE))
        self.opt = dict(graph.meta.get("optimizer", {"kind": "none"}))
        self.lr_fn: Optional[Callable[[int], float]] = None
        self.lr_now = 0.0
        _spec = (graph.meta.get("optimizer") or {}).get("schedule")
        if _spec:      # a schedule that came with the graph (e.g. from a client over RPC); Trainer.set_lr_schedule overrides it
            from ..utils.schedules import from_spec
            self.lr_fn = from_spec(_spec, (graph.meta.get("optimizer") or {}).get("lr") or 0.0)
        self._plan()

    # ------------------------------------------------------------------ planning
    def _plan(self) -> None:
        g = self.g
        last_use: Dict[Tuple[int, int], int] = {}
        for n in g.nodes:
            for v in n.inputs:
                last_use[v.key()] = n.id
        for v in g.outputs:
            last_use[v.key()] = len(g.nodes)
        self.free_after: Dict[int, List[Tuple[int, int]]] = {}
        for k, nid in last_use.items():
            if nid < len(g.nodes):
                self.free_after.setdefault(nid, []).append(k)
        # gradient values feeding apply_* nodes are bound to the flat gradient buffer
        self.grad_binding: Dict[Tuple[int, int], int] = {}
        self.apply_nodes: List[Node] = [n for n in g.nodes if n.op.startswith("apply_")]
        for n in self.apply_nodes:
            pid = n.inputs[0].node
            if g.nodes[pid].op == "parameter":
                self.grad_binding[n.inputs[1].key()] = pid
        self.first_apply = self.apply_nodes[0].id if self.apply_nodes else None
        if any(len(n.inputs) > 2 for n in self.apply_nodes):
            self.store.ensure_slots(flat_moments=any(n.op == "apply_adamw" for n in self.apply_nodes))
        # nodes that (transitively) consume an optimizer output run after the update phase
        self.post_apply: set = set()
        for n in g.nodes:
            if n.op.startswith("apply_") or any(v.node in self.post_apply for v in n.inputs):
                self.post_apply.add(n.id)
        # the flat fused update needs every apply node to act on whole variables laid out like the flat buffers
        def _whole(n):
            if g.nodes[n.inputs[0].node].op != "parameter":
                return False
            return all(g.nodes[v.node].op == "state" and tuple(g.type_of(v).shape) == tuple(g.type_of(n.inputs[0]).shape)
                       for v in n.inputs[2:])
        # gradient clipping (reference examples/gpt_moe/optimizers/__init__.py:150-159: clip_by_norm per tensor / clip_by_global_norm):
        # needs every gradient in its final form before any update starts, so the updates run per variable on the general
        # path (no flat fused / sharded-optimizer kernels, which consume gradients bucket by bucket during backward)
        self.clip: Optional[Tuple[str, float]] = None
        if self.opt.get("clip_norm"):
            if self.opt["clip_norm"] not in ("global", "local"):
                raise ValueError(f"clip_norm={self.opt['clip_norm']!r}: expected 'global' or 'local'")
            self.clip = (self.opt["clip_norm"], float(self.opt.get("clip_norm_value", 1.0)))
        self._clip_scales: Dict[int, torch.Tensor] = {}
        self.pipeline_norm_divisor = 0       # set by a pipeline stage worker: SPMD replicas per stage (0 = not a pipeline)
        self.fused_apply_ok = self.clip is None and all(_whole(n) and n.op in FLAT_APPLY for n in self.apply_nodes)
        if not self.fused_apply_ok:
            self.grad_binding = {}  # general path: gradients flow through the environment, not the flat buffer
        self.update_target: Dict[Tuple[int, int], int] = {v.key(): var for var, v in g.updates.items()}
        self.flat_zero: Optional[Dict[str, Any]] = None
        if self._fz_static is not None and self.collective is not None:
            self._detect_flat_zero()
        # where each variable's moments really live (see VariableStore.flat_moment_pids)
        if not (self.fused_apply_ok and self.flat_zero is None):
            flat = {n_.attrs.get("slot_of") for n_ in self.store._state_nodes if self.store._flat_slot(n_)}
            if self.flat_zero is not None:
                def _root(v):
                    nd_ = g.nodes[v.node]
                    while nd_.op == "dynamic_slice":
                        nd_ = g.nodes[nd_.inputs[0].node]
                    return nd_.id
                flat |= {_root(g.nodes[aid].inputs[0]) for aid in self.flat_zero["regular_apply"]}
                flat |= {pid_ for (pid_, _, _, _) in (self.flat_zero.get("replicated_apply") or {}).values()}
            self.store.flat_moment_pids = flat
        # peephole: dX_total = add(dX_residual, layernorm_bwd.dx) -> the LN-backward kernel adds the residual gradient
        self.ln_fuse: Dict[int, Tuple[int, int]] = {}
        self.alias_of: Dict[int, Tuple[int, int]] = {}
        users = g.users()
        for n in g.nodes:
            if n.op != "add" or len(n.inputs) != 2:
                continue
            for k in (0, 1):
                v, o = n.inputs[k], n.inputs[1 - k]
                p_ = g.nodes[v.node]
                if (p_.op == "layernorm_bwd" and v.idx == 0 and len(users.get(v.key(), [])) == 1 and o.node < p_.id
                        and tuple(g.type_of(o).shape) == tuple(g.type_of(v).shape) and p_.id not in self.ln_fuse
                        and v.key() not in {x.key() for x in g.outputs}):
                    self.ln_fuse[p_.id] = o.key()
                    self.alias_of[n.id] = v.key()
                    last_use[o.key()] = max(last_use.get(o.key(), 0), p_.id)
                    break
        # peephole: gelu(linear(x)) -> one GEMM writing pre-activation + activation; gelu_bwd(linear_dgrad(dz), f) ->
        # the dgrad GEMM multiplies by GELU'(f) in its epilogue (GPU only: these are epilogues of the tcgen05 kernel)
        self.gelu_dual: Dict[int, int] = {}
        self.gelu_bwd_fuse: Dict[int, Tuple[int, int]] = {}
        if self.device.type == "cuda":
            for n in g.nodes:
                if n.op == "gelu":
                    v = n.inputs[0]
                    L = g.nodes[v.node]
                    us = users.get(v.key(), [])
                    if (L.op == "linear" and not L.attrs.get("residual") and L.id not in self.gelu_dual
                            and all(g.nodes[u].op in ("gelu", "gelu_bwd") for u, _ in us) and sum(g.nodes[u].op == "gelu" for u, _ in us) == 1
                            and g.type_of(v).dtype == "bf16"):
                        self.gelu_dual[L.id] = n.id
                        self.alias_of[n.id] = (L.id, 1)
                        last_use[(L.id, 1)] = last_use.get((n.id, 0), n.id)
                elif n.op == "gelu_bwd":
                    dy, f = n.inputs
                    D = g.nodes[dy.node]
                    if (D.op == "linear_dgrad" and len(users.get(dy.key(), [])) == 1 and f.node < D.id and D.id not in self.gelu_bwd_fuse
                            and g.type_of(dy).dtype == "bf16"):
                        self.gelu_bwd_fuse[D.id] = f.key()
                        self.alias_of[n.id] = dy.key()
                        last_use[f.key()] = max(last_use.get(f.key(), 0), n.id)
        self.free_after = {}
        for k_, nid in last_use.items():
            if nid < len(g.nodes):
                self.free_after.setdefault(nid, []).append(k_)
        self.ln_stats: Dict[Tuple[Tuple[int, int], Tuple[int, int]], Tuple[torch.Tensor, torch.Tensor]] = {}
        self.bn_stats: Dict[Tuple[int, Tuple[int, int]], Tuple[torch.Tensor, torch.Tensor]] = {}
        self.bn_sync_stats: Dict[Tuple[int, Tuple[int, int]], Tuple[torch.Tensor, torch.Tensor]] = {}
        self.input_names = [n.name for n in g.inputs()]
        self.grad_accumulate = False   # True when gradients add up over micro-batches (pipeline stage workers)
        self._plan_store_init()
        self.tp_fuse: Dict[int, Dict[str, Any]] = {}
        self._moe_routes: Dict[Tuple[Any, int], Dict[str, Any]] = {}
        self._moe_einsum: Dict[int, Tuple[str, int]] = self._find_moe_einsums(self.g) if MOE_SPARSE else {}
        if TP_FUSED and self.collective is not None and ((self.comm_mode == "fused" and self.device.type == "cuda") or TP_FUSED_IMPL):
            self._plan_tp_fusion()

    @staticmethod
    def _analyze_flat_zero(g: Graph) -> Optional[Dict[str, Any]]:
        """Recognise the planner's data-parallel optimizer pattern
              grad -> {reduce_scatter | all_reduce}(level L) -> apply(param or dynamic_slice(param), slots...) [-> all_gather -> update]
        Variables that follow it ("regular") are executed over the FLAT buffers: bucketed reduce-scatter of the gradient
        buffer (launched as soon as a bucket's last gradient exists, overlapping the rest of backward), one fused AdamW
        over the owned chunks, one all-gather of the bf16 parameters per bucket.  This is the combiner (SURVEY B7) taken
        to its conclusion; the per-tensor collectives of the plan become virtual.  Variables the planner treated
        differently (stored sharded, gradient re-laid-out by all-to-all, ...) keep the general per-tensor path."""
        apply_nodes = [n for n in g.nodes if n.op.startswith("apply_")]
        if not apply_nodes or any(n.op not in FLAT_APPLY for n in apply_nodes) or (g.meta.get("optimizer") or {}).get("clip_norm"):
            return None     # (optimizers with per-variable reductions cannot be applied over flat, variable-straddling chunks;
                            #  gradient clipping needs all gradients before the first update)
        skip: set = set()
        binding: Dict[Tuple[int, int], int] = {}
        regular_apply: set = set()
        irregular_params: set = set()
        replicated: Dict[int, Tuple[int, Tuple[int, int]]] = {}   # apply node -> (param, gradient value)
        level = num = None
        for a in apply_nodes:
            nd = g.nodes[a.inputs[0].node]
            local_skip = set()
            if nd.op == "parameter":
                pid = nd.id
            elif nd.op == "dynamic_slice" and g.nodes[nd.inputs[0].node].op == "parameter":
                pid = nd.inputs[0].node
                local_skip.add(nd.id)
            else:
                pid = None
            c = g.nodes[a.inputs[1].node]
            ok = pid is not None and c.op in ("reduce_scatter", "all_reduce")
            if ok:
                # the variable must be stored whole (a shard-shaped parameter is a different ownership scheme)
                ok = "shard_dims" not in g.nodes[pid].attrs
            if ok:
                l, k = int(c.attrs["level"]), int(c.attrs["num"])
                if level is None:
                    level, num = l, k
                ok = (level, num) == (l, k)
            if not ok:
                root = nd.id if nd.op == "parameter" else (nd.inputs[0].node if nd.inputs else None)
                if root is not None and g.nodes[root].op == "parameter":
                    irregular_params.add(root)
                    # whole variable, whole slots, gradient computed redundantly on every rank (no collective in front of
                    # the apply): the update can still be sharded -- owner updates its chunk and stores it to every peer
                    if (nd.op == "parameter" and c.op not in COLLECTIVE_OPS and "shard_dims" not in nd.attrs
                            and all(g.nodes[v.node].op == "state" for v in a.inputs[2:])):
                        replicated[a.id] = (root, a.inputs[1].key())
                continue
            binding[c.inputs[0].key()] = pid
            regular_apply.add(a.id)
            skip |= local_skip
            skip.add(c.id)
            for v in a.inputs[2:]:
                if g.nodes[v.node].op == "dynamic_slice":
                    skip.add(v.node)
        if level is None or num <= 1 or not regular_apply:
            return None
        # post-update nodes (all-gathers of updated shards ...) that only serve regular variables are virtual too
        anc: Dict[int, set] = {}
        for n in g.nodes:
            s_: set = set()
            if n.op.startswith("apply_"):
                s_.add(n.id)
            for v in n.inputs:
                s_ |= anc.get(v.node, set())
            if s_:
                anc[n.id] = s_
                if not n.op.startswith("apply_") and s_ <= regular_apply:
                    skip.add(n.id)
        return {"level": level, "num": num, "skip": skip, "binding": binding, "regular_apply": regular_apply,
                "irregular_params": irregular_params, "replicated": replicated}

    def _detect_flat_zero(self) -> None:
        fz = self._fz_static
        if fz is None:
            return
        g, st = self.g, self.store
        if self.opt.get("kind") == "adamw":
            st.ensure_slots(flat_moments=True)      # the chunked update addresses m / v by flat offset
        num = fz["num"]
        bucket_elems = int(self.opt.get("bucket_elems", 48 * 1024 * 1024))
        gran = num * _ALIGN
        end = (st.regular_end + gran - 1) // gran * gran
        if end > st.regular_end:
            if st.regular_end != st.total:   # irregular tail present: cannot pad in the middle -> shift is not
                # needed because every offset is _ALIGN aligned; pad only matters at the very end of the range
                end = st.regular_end // gran * gran
            else:
                st.grow(end)
        offs = sorted((st.offset[p], p) for p in st.order if p not in fz["irregular_params"])
        tail_regular = [(o, p) for o, p in offs if o >= end]          # regular variables beyond the aligned range
        offs = [(o, p) for o, p in offs if o < end]
        if not offs:
            return
        # graded bucket sizes: the variables at the front of the flat buffer belong to the first layers, whose gradients
        # are produced LAST by the backward pass -- whatever is still in flight when backward ends is exposed, so the
        # buckets that become ready last are small (4M elements, doubling up to bucket_elems)
        first = int(self.opt.get("first_bucket_elems", os.environ.get("TEPDIST_FIRST_BUCKET", 4 * 1024 * 1024)))
        from .. import _C
        # (the bucket policy lives in the C++ core next to the gradient-collective combiner: csrc/transform.cc PlanFlatBuckets)
        bounds = list(_C.plan_flat_buckets([int(off) for off, _ in offs], int(end), int(gran), int(first), int(bucket_elems)))
        buckets = [(bounds[i], bounds[i + 1]) for i in range(len(bounds) - 1)]
        binding = {k: v for k, v in fz["binding"].items()}
        regular_apply = set(fz["regular_apply"])
        skip = set(fz["skip"])
        if tail_regular:   # (a partially covered variable cannot be split across ownership schemes)
            cut = {p for _, p in tail_regular}
            # variables straddling `end` also fall back
            for o, p in offs:
                n_el = 1
                for d in st.shape[p]:
                    n_el *= d
                if o + n_el > end:
                    cut.add(p)
            if cut:
                self._fz_static = None
                return
        prod_of_param = {pid: key[0] for key, pid in binding.items()}
        ready_at: Dict[int, List[int]] = {}
        for bi, (s0, e0) in enumerate(buckets):
            last = max((prod_of_param[p] for off, p in offs if s0 <= off < e0 and p in prod_of_param), default=-1)
            ready_at.setdefault(last, []).append(bi)
        self.grad_binding = binding
        self.flat_zero = {"level": fz["level"], "num": num, "skip": skip, "buckets": buckets, "ready_at": ready_at,
                          "rank": self.coords.get(fz["level"], 0), "regular_apply": regular_apply, "fused": None}
        # replicated-gradient variables (e.g. embeddings whose backward the plan replicates on every rank): the gradient
        # lands in the flat buffer and the UPDATE is still sharded -- the owner updates its chunk from the local gradient
        # and publishes it (fused mode: P2P stores from the same kernel; NCCL mode: all-gather).  (N-1)/N less AdamW
        # traffic, and the replicas stay bit-identical (redundant fp32 atomics would let them drift apart).
        rep = {}
        if self.opt.get("kind") == "adamw" and st.m is not None:
            for aid, (pid, gkey) in fz.get("replicated", {}).items():
                n_el = 1
                for d in st.shape[pid]:
                    n_el *= d
                if n_el % (4 * num) == 0 and st.offset[pid] % 4 == 0 and g.nodes[aid].op == "apply_adamw":
                    rep[aid] = (pid, st.offset[pid], n_el, bool(g.nodes[aid].attrs.get("decay", True)))
                    self.grad_binding[gkey] = pid
        self.flat_zero["replicated_apply"] = rep
        if (self.comm_mode == "fused" and st.master.is_cuda and self.opt.get("kind") == "adamw" and num <= 8):
            from ..parallel.symm import FusedShardedOptimizer
            pg = self.collective.mesh.group(fz["level"])
            try:
                st.make_symmetric(pg)
                self.flat_zero["fused"] = FusedShardedOptimizer(st.symm_grad, st.symm_param, pg, grad16_buf=st.symm_grad16)
                self.flat_zero["fused"].dry = self.dry_comm
            except RuntimeError as e:   # e.g. CUDA IPC unavailable in this container: keep the NCCL path, loudly
                import warnings
                warnings.warn(f"fused peer-memory optimizer unavailable ({e}); falling back to NCCL collectives")
                self.flat_zero["fused"] = None
                self.comm_mode = "nccl"
        self.fused_apply_ok = True  # regular gradients land in the flat buffer again

    def _flat_zero_reduce(self, bi: int, pending: List[Any]) -> None:
        import torch.distributed as dist
        fz, st = self.flat_zero, self.store
        if fz["fused"] is not None:
            # fused mode: as soon as the bucket's gradients exist, a side stream runs
            #   barrier -> [P2P reduce-scatter + AdamW + bf16 P2P all-gather] for this bucket
            # with a small CTA budget so it overlaps the remaining backward GEMMs instead of displacing them
            fo, o = fz["fused"], self.opt
            if fz.get("comm_stream") is None:
                fz["comm_stream"] = torch.cuda.Stream()
            cs = fz["comm_stream"]
            cs.wait_stream(torch.cuda.current_stream())
            s0, e0 = fz["buckets"][bi]
            n, r = fz["num"], fz["rank"]
            chunk = (e0 - s0) // n
            last = len(pending) == len(fz["buckets"]) - 1
            with torch.cuda.stream(cs):
                if fo.g16 is not None and not fo.dry:      # bf16 wire: stage this bucket's gradients (all of it: peers reduce their chunks of it)
                    ops.cast_f32_bf16(st.grad[s0:e0], fo.g16.tensor(torch.bfloat16, st.total)[s0:e0])
                fo.barrier()
                fo.step(st.master, st.m, st.v, s0 + r * chunk, s0 + (r + 1) * chunk, st.n_decay, self.hyper,
                        o.get("beta1", 0.9), o.get("beta2", 0.999), o.get("eps", 1e-8), o.get("weight_decay", 0.0),
                        ctas=0 if last else int(os.environ.get("TEPDIST_OVERLAP_CTAS", o.get("overlap_ctas", 74))))   # 74: measured A/B on 4 x B200, 16.89 vs 17.37 ms with 296 (37: 17.88)
            pending.append(None)
            return
        s0, e0 = fz["buckets"][bi]
        n, r = fz["num"], fz["rank"]
        chunk = (e0 - s0) // n
        pg = self.collective.mesh.group(fz["level"])
        buf = st.grad[s0:e0]
        own = st.grad[s0 + r * chunk:s0 + (r + 1) * chunk]
        if self.dry_comm:
            pending.append(None)
        elif buf.is_cuda:
            pending.append(dist.reduce_scatter_tensor(own, buf, group=pg, async_op=True))
        else:  # gloo has no reduce-scatter
            pending.append(dist.all_reduce(buf, group=pg, async_op=True))

    def _flat_zero_apply(self, pending: List[Any]) -> None:
        import torch.distributed as dist
        fz, st, o = self.flat_zero, self.store, self.opt
        n, r = fz["num"], fz["rank"]
        if fz["fused"] is not None:
            fo = fz["fused"]
            cs = fz.get("comm_stream")
            rep = fz.get("replicated_apply") or {}
            if cs is None and rep:
                cs = fz["comm_stream"] = torch.cuda.Stream()
            if cs is not None:
                if rep:
                    cs.wait_stream(torch.cuda.current_stream())     # their gradients are the last thing backward produces
                with torch.cuda.stream(cs):
                    for aid, (pid, off, n_el, decay) in rep.items():
                        chunk = n_el // n
                        fo.step(st.master, st.m, st.v, off + r * chunk, off + (r + 1) * chunk, off + n_el if decay else off,
                                self.hyper, o.get("beta1", 0.9), o.get("beta2", 0.999), o.get("eps", 1e-8),
                                o.get("weight_decay", 0.0), ctas=0, local_grad=True)
                    fo.barrier()    # every rank's parameter shards have landed everywhere
                torch.cuda.current_stream().wait_stream(cs)
            return
        for w in pending:
            if w is not None:
                w.wait()
        pg = self.collective.mesh.group(fz["level"])
        works = []
        for (s0, e0) in fz["buckets"]:
            chunk = (e0 - s0) // n
            a, b = s0 + r * chunk, s0 + (r + 1) * chunk
            nd = min(max(st.n_decay - a, 0), b - a)
            kind = o.get("kind")
            comp = None if st.compute is None else st.compute[a:b]
            if kind == "adamw":
                ops.adamw_step(st.master[a:b], st.grad[a:b], st.m[a:b], st.v[a:b], comp, nd, self._lr(1e-3),
                               o.get("beta1", 0.9), o.get("beta2", 0.999), o.get("eps", 1e-8), o.get("weight_decay", 0.0),
                               self.step_count, hyper=self.hyper if st.master.is_cuda else None)
            elif kind == "sgd":
                ops.sgd_step(st.master[a:b], st.grad[a:b], comp, self._lr(1e-2))
            tgt = st.compute if st.compute is not None else st.master
            if not self.dry_comm:
                works.append(dist.all_gather_into_tensor(tgt[s0:e0], tgt[a:b], group=pg, async_op=True))
        for aid, (pid, off, n_el, decay) in (fz.get("replicated_apply") or {}).items():
            chunk = n_el // n
            a, b = off + r * chunk, off + (r + 1) * chunk
            comp = None if st.compute is None else st.compute[a:b]
            ops.adamw_step(st.master[a:b], st.grad[a:b], st.m[a:b], st.v[a:b], comp, (b - a) if decay else 0, self._lr(1e-3),
                           o.get("beta1", 0.9), o.get("beta2", 0.999), o.get("eps", 1e-8), o.get("weight_decay", 0.0),
                           self.step_count, hyper=self.hyper if st.master.is_cuda else None)
            tgt = st.compute if st.compute is not None else st.master
            if not self.dry_comm:
                works.append(dist.all_gather_into_tensor(tgt[off:off + n_el], tgt[a:b], group=pg, async_op=True))
        for w in works:
            w.wait()

    def materialize_full_state(self) -> None:
        """ZeRO-style execution updates the fp32 master weights and moments only in the chunk each rank owns; outside it
        they go stale (only the bf16 compute copy is all-gathered every step).  Before a checkpoint / state_dict every rank
        gathers the owners' chunks so master, m and v are whole and identical everywhere.  Collective: all ranks call it."""
        fz = self.flat_zero
        if fz is None:
            return
        import torch.distributed as dist
        st = self.store
        n, r = fz["num"], fz["rank"]
        pg = self.collective.mesh.group(fz["level"])
        ranges = [(s0, e0) for (s0, e0) in fz["buckets"]]
        ranges += [(off, off + n_el) for (_, off, n_el, _) in (fz.get("replicated_apply") or {}).values()]
        if st.master.is_cuda:
            torch.cuda.synchronize()
        for buf in (st.master, st.m, st.v):
            if buf is None:
                continue
            for (s0, e0) in ranges:
                chunk = (e0 - s0) // n
                dist.all_gather_into_tensor(buf[s0:e0], buf[s0 + r * chunk:s0 + (r + 1) * chunk].clone(), group=pg)

    # ------------------------------------------------------------------ running
    def step(self, feeds: Dict[str, torch.Tensor]) -> List[torch.Tensor]:
        self.step_count += 1
        self._set_hyper()
        if not self.use_cuda_graph:
            return self._run(feeds)
        if self._graph is None:
            if not self._static_in:
                # first call: static input buffers + an eager step on a side stream (it is both this call's step and the
                # warm-up the capture needs: lazy allocations, symmetric buffers, kernel attribute setup)
                for k, t in feeds.items():
                    self._static_in[k] = t.to(self.device).clone()
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    out = self._run(self._static_in)
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize()
                return out
            # second call: capture, then replay once -- exactly ONE optimizer update per step() call (an eager run followed by
            # capture + replay would apply the same batch twice with the same step index)
            for k, t in feeds.items():
                self._static_in[k].copy_(t, non_blocking=True)
            torch.cuda.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._static_out = self._run(self._static_in)
            self._launches_per_step = self._last_launches
            self._graph.replay()  # capture records but does not execute: run the recorded step now
            ops._count(self._launches_per_step)
            return self._static_out
        for k, t in feeds.items():
            self._static_in[k].copy_(t, non_blocking=True)
        self._graph.replay()
        ops._count(self._launches_per_step)
        return self._static_out

    def _set_hyper(self) -> None:
        kind = self.opt.get("kind")
        lr = self.lr_fn(self.step_count) if self.lr_fn else self.opt.get("lr", 1e-3)
        lr = 0.0 if lr is None else float(lr)      # (lr=None: Adafactor's relative step size, hyper[H_AF_REL_LR])
        self.lr_now = lr
        from .optimizers import host_hyper
        vals = host_hyper(self.opt, self.step_count, lr)
        if kind is None:
            return
        for i, x in enumerate(vals):
            self._hyper_host[i] = x
        self.hyper.copy_(self._hyper_host, non_blocking=True)

    def _lr(self, default: float) -> float:
        """Learning rate for the update paths that take it as a host scalar (CPU fallbacks, the SGD kernel): the schedule's
        value of this step when one is set, else the graph's constant.  (The AdamW kernels and the torch-op optimizers read
        hyper[0] on the device instead, which is what keeps a schedule working under CUDA-graph replay.)"""
        return self.lr_now if self.lr_fn is not None else self.opt.get("lr", default)

    def set_lr_schedule(self, fn: Optional[Callable[[int], float]]) -> None:
        """`fn(step)` -> learning rate of optimizer step `step` (1-based); None restores the graph's constant."""
        if fn is not None and self.use_cuda_graph and self.opt.get("kind") == "sgd" and self.device.type == "cuda":
            raise NotImplementedError("a learning-rate schedule with SGD under CUDA-graph replay: the SGD kernel takes the rate as a "
                                      "launch argument, which a captured graph freezes; use use_cuda_graph=False or AdamW / momentum")
        self.lr_fn = fn

    def _run(self, feeds: Dict[str, torch.Tensor]) -> List[torch.Tensor]:
        g = self.g
        env: Dict[Tuple[int, int], torch.Tensor] = {}
        self._zero_grads()  # GAInit
        launches0 = ops.launch_count()

        def run_node(n: Node) -> None:
            self._run_node(n, env, feeds)

        fz = self.flat_zero
        pending: List[Any] = []
        if fz is not None and -1 in fz["ready_at"]:
            for bi in fz["ready_at"][-1]:
                self._flat_zero_reduce(bi, pending)
        for n in g.nodes:
            if n.op == "state" or n.id in self.post_apply:
                continue
            if fz is not None and n.id in fz["skip"]:
                continue
            run_node(n)
            if fz is not None and n.id in fz["ready_at"]:
                for bi in fz["ready_at"][n.id]:
                    self._flat_zero_reduce(bi, pending)   # overlaps with the remaining backward kernels
        self.run_optimizer(env, feeds, pending if fz is not None else None)
        self._last_launches = ops.launch_count() - launches0
        return [env[v.key()] for v in g.outputs]

    def _run_node(self, n: Node, env: Dict[Tuple[int, int], torch.Tensor], feeds: Dict[str, torch.Tensor]) -> None:
        g = self.g
        if n.id in self.alias_of:        # fused into the producer (see ln_fuse)
            outs = [env[self.alias_of[n.id]]]
        else:
            ins = [env[v.key()] for v in n.inputs]
            self._env = env
            prof = getattr(self, "_prof", None)
            if prof is None or n.op in SOURCE_OPS:
                outs = self._exec(n, ins, feeds)
            else:
                t0 = self._prof_mark()
                outs = self._exec(n, ins, feeds)
                prof.append((n.name or f"{n.op}_{n.id}", n.op, t0, self._prof_mark()))
        for i, t in enumerate(outs):
            env[(n.id, i)] = t
            pid = self.grad_binding.get((n.id, i))
            if pid is not None and self.fused_apply_ok:  # a variable's final gradient lands in the flat buffer
                gv = self.store.grad_view(pid)
                if t.data_ptr() != gv.data_ptr():
                    gv.add_(t.reshape(gv.shape).to(gv.dtype))
            var = self.update_target.get((n.id, i))
            if var is not None and g.nodes[var].op == "parameter":  # e.g. all-gathered updated shards
                dst = self.store.compute_view(var)
                if t.data_ptr() != dst.data_ptr():
                    dst.copy_(t.reshape(dst.shape))
        for k in self.free_after.get(n.id, ()):
            if k not in self.grad_binding:
                env.pop(k, None)

    # ------------------------------------------------------------------ profiling (reference: per-task timing under DEBUG,
    # virtual_client.cc:1672,1700-1702 -- host wall clock there, device events here)
    def _prof_mark(self):
        if self.device.type == "cuda":
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            return e
        import time
        return time.perf_counter()

    def profile(self, feeds: Dict[str, torch.Tensor], warmup: int = 1, chrome_trace: Optional[str] = None) -> Dict[str, Any]:
        """Run one EAGER step with a device timestamp on both sides of every node and return the time per node and per
        op kind (ms).  Nodes on side streams (overlapped optimizer buckets) are attributed to the launch position.
        `chrome_trace`: also write a chrome://tracing JSON timeline."""
        feeds = {k: t.to(self.device) for k, t in feeds.items()}
        for _ in range(warmup):
            self.step_count += 1
            self._set_hyper()
            self._run(feeds)
        self.step_count += 1
        self._set_hyper()
        self._prof = []
        start = self._prof_mark()
        try:
            self._run(feeds)
            end = self._prof_mark()
            if self.device.type == "cuda":
                torch.cuda.synchronize()
            rec = self._prof
        finally:
            self._prof = None
        ms = (lambda a, b: a.elapsed_time(b)) if self.device.type == "cuda" else (lambda a, b: (b - a) * 1e3)
        nodes = [{"name": nm, "op": op, "start_ms": ms(start, t0), "ms": ms(t0, t1)} for nm, op, t0, t1 in rec]
        by_op: Dict[str, float] = {}
        for r in nodes:
            by_op[r["op"]] = by_op.get(r["op"], 0.0) + r["ms"]
        out = {"total_ms": ms(start, end), "by_op": dict(sorted(by_op.items(), key=lambda kv: -kv[1])), "nodes": nodes}
        if chrome_trace:
            import json
            ev = [{"name": r["name"], "cat": r["op"], "ph": "X", "pid": 0, "tid": 0, "ts": r["start_ms"] * 1e3,
                   "dur": r["ms"] * 1e3} for r in nodes]
            with open(chrome_trace, "w") as f:
                json.dump({"traceEvents": ev, "displayTimeUnit": "ms"}, f)
        return out

    def run_optimizer(self, env: Dict[Tuple[int, int], torch.Tensor], feeds: Dict[str, torch.Tensor], pending: Optional[List[Any]] = None) -> None:
        """Gradient sync + optimizer update + post-update nodes, for whichever execution scheme is active."""
        g, fz = self.g, self.flat_zero
        if not self.apply_nodes:
            return
        prof = getattr(self, "_prof", None)
        if prof is not None:
            t0 = self._prof_mark()
            self._prof = None
            try:
                self.run_optimizer(env, feeds, pending)
            finally:
                self._prof = prof
            prof.append(("optimizer(+grad sync)", "optimizer", t0, self._prof_mark()))
            return
        if fz is not None:
            if pending is None:
                pending = []
                for bi in range(len(fz["buckets"])):
                    self._flat_zero_reduce(bi, pending)
            self._flat_zero_apply(pending)
            done = fz.get("replicated_apply") or {}
            for n in self.apply_nodes:
                if n.id not in fz["regular_apply"] and n.id not in done:
                    self._apply_one(n, env)
            for n in g.nodes:
                if n.id in self.post_apply and not n.op.startswith("apply_") and n.id not in fz["skip"]:
                    self._run_node(n, env, feeds)
            return
        if self.grad_sync is not None:
            self.grad_sync(self.store.grad)
        if self.fused_apply_ok:
            self._fused_apply()
            for n in self.apply_nodes:
                env[(n.id, 0)] = self.store.compute_view(n.inputs[0].node)
        else:
            if self.clip is not None:
                self._compute_clip_scales(env)
            for n in self.apply_nodes:
                self._apply_one(n, env)
        for n in g.nodes:
            if n.id in self.post_apply and not n.op.startswith("apply_"):
                self._run_node(n, env, feeds)

    def _shard_chain(self, v: Value) -> List[Tuple[int, int, int]]:
        """[(dim, num, level)] that cut this rank's view `v` (a variable or dynamic_slices of one) out of the full variable."""
        g = self.g
        chain: List[Tuple[int, int, int]] = []
        src = g.nodes[v.node]
        while src.op == "dynamic_slice":
            chain.insert(0, (int(src.attrs["dim"]), int(src.attrs["num"]), int(src.attrs["level"])))
            src = g.nodes[src.inputs[0].node]
        return [(int(d_), int(k_), int(l_)) for d_, k_, l_ in zip(src.attrs.get("shard_dims", []), src.attrs.get("shard_nums", []),
                                                                  src.attrs.get("shard_levels", []))] + chain

    def _compute_clip_scales(self, env: Dict[Tuple[int, int], torch.Tensor]) -> None:
        """Per apply node: the factor its gradient is multiplied with.  'global': min(1, c / |all gradients|), 'local':
        min(1, c / |this gradient|).  Norms are over WHOLE variables: a gradient that is a shard of its variable contributes its
        local sum of squares, completed over the levels that shard it (one all-reduce per distinct set of levels); pipeline
        stages add theirs up over the whole job.  Device tensors throughout: nothing synchronises, the step stays capturable."""
        import torch.distributed as dist
        mode, c = self.clip
        live = self.collective is not None and not self.collective.dry and self.collective.mesh.world > 1
        sq: Dict[int, torch.Tensor] = {}
        by_levels: Dict[Tuple[int, ...], List[int]] = {}
        for n in self.apply_nodes:
            gr = env[n.inputs[1].key()].float()
            sq[n.id] = (gr * gr).sum().reshape(1)
            lv = tuple(sorted({l for _, k, l in self._shard_chain(n.inputs[0]) if k > 1})) if live else ()
            by_levels.setdefault(lv, []).append(n.id)
        for lv, ids in by_levels.items():
            if lv:
                t = torch.cat([sq[i] for i in ids])
                for l in lv:
                    dist.all_reduce(t, group=self.collective.mesh.group(l))
                for j, i in enumerate(ids):
                    sq[i] = t[j:j + 1]
        if mode == "local":
            for n in self.apply_nodes:
                self._clip_scales[n.id] = torch.clamp(c / (torch.sqrt(sq[n.id]) + 1e-6), max=1.0).reshape(())
            return
        total = torch.cat(list(sq.values())).sum().reshape(1)
        if self.pipeline_norm_divisor and dist.is_initialized():
            total = total / float(self.pipeline_norm_divisor)     # every SPMD replica of a stage holds the stage's full sum
            dist.all_reduce(total)
        scale = torch.clamp(c / (torch.sqrt(total) + 1e-6), max=1.0).reshape(())
        for n in self.apply_nodes:
            self._clip_scales[n.id] = scale

    def _apply_one(self, n: Node, env: Dict[Tuple[int, int], torch.Tensor]) -> None:
        """General (un-fused) optimizer update of one variable or one shard of it (ZeRO-style plans: the update acts
        on dynamic_slice(parameter) with sharded slots; the updated shard is all-gathered by a later node)."""
        g, st, o = self.g, self.store, self.opt
        grad = env[n.inputs[1].key()].float().contiguous()
        if self.clip is not None:
            grad = grad * self._clip_scales[n.id]

        def storage(v: Value, which: str) -> torch.Tensor:
            """Persistent storage behind `v` (a variable/slot, or this rank's dynamic_slice of one)."""
            src = g.nodes[v.node]
            def base(nd):
                if nd.op == "parameter":
                    return st.master_view(nd.id) if which == "master" else st.compute_view(nd.id)
                assert nd.op == "state", nd.op
                return st.state[nd.id]
            if src.op in ("parameter", "state"):
                return base(src)
            assert src.op == "dynamic_slice", src.op
            b = storage(src.inputs[0], which)       # (nested: one dynamic_slice per mesh level that shards the variable)
            d, num = int(src.attrs["dim"]), int(src.attrs["num"])
            sz = b.shape[d] // num
            return b.narrow(d, self.coords.get(int(src.attrs["level"]), 0) * sz, sz)

        master = storage(n.inputs[0], "master")
        comp = storage(n.inputs[0], "compute")
        if n.op not in FLAT_APPLY:
            # optimizers with per-variable reductions (runtime/optimizers.py): in place on this rank's view, reductions
            # completed over the mesh levels that cut the view out of the variable
            from .optimizers import STEP, Shards
            chain: List[Tuple[int, int, int]] = []
            src = g.nodes[n.inputs[0].node]
            while src.op == "dynamic_slice":
                chain.insert(0, (int(src.attrs["dim"]), int(src.attrs["num"]), int(src.attrs["level"])))
                src = g.nodes[src.inputs[0].node]
            chain = [(int(d_), int(k_), int(l_)) for d_, k_, l_ in zip(src.attrs.get("shard_dims", []), src.attrs.get("shard_nums", []),
                                                                       src.attrs.get("shard_levels", []))] + chain

            def all_reduce(t: torch.Tensor, level: int, op: str) -> None:
                if self.collective is None or self.collective.dry or self.collective.mesh.world == 1:
                    return
                import torch.distributed as dist
                dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM, group=self.collective.mesh.group(level))
            slots = [storage(v, "state") for v in n.inputs[2:]]
            STEP[n.op](master, grad.reshape(master.shape), slots, o, self.hyper, Shards(chain, all_reduce), decay=bool(n.attrs.get("decay", True)))
            if comp.data_ptr() != master.data_ptr():
                comp.copy_(master.to(comp.dtype))
            env[(n.id, 0)] = comp if comp.is_contiguous() else comp.contiguous()
            for i, sl in enumerate(slots):
                env[(n.id, i + 1)] = sl
            return
        pm = master if master.is_contiguous() else master.contiguous()
        pc = comp if (comp.is_contiguous() and comp.dtype == torch.bfloat16) else (
            torch.empty(pm.shape, dtype=torch.bfloat16, device=pm.device) if pm.is_cuda else None)
        decay = bool(n.attrs.get("decay", True))
        if n.op == "apply_adamw":
            m_st, v_st = storage(n.inputs[2], "state"), storage(n.inputs[3], "state")
            m = m_st if m_st.is_contiguous() else m_st.contiguous()
            v = v_st if v_st.is_contiguous() else v_st.contiguous()
            numel = pm.numel()
            ops.adamw_step(pm.view(-1), grad.view(-1), m.view(-1), v.view(-1), None if pc is None else pc.view(-1),
                           numel if decay else 0, self._lr(1e-3), o.get("beta1", 0.9), o.get("beta2", 0.999),
                           o.get("eps", 1e-8), o.get("weight_decay", 0.0), self.step_count,
                           hyper=self.hyper if pm.is_cuda else None)
            if m.data_ptr() != m_st.data_ptr():
                m_st.copy_(m); v_st.copy_(v)
            env[(n.id, 1)], env[(n.id, 2)] = m, v
        else:
            ops.sgd_step(pm.view(-1), grad.view(-1), None if pc is None else pc.view(-1), self._lr(1e-2))
        if pm.data_ptr() != master.data_ptr():
            master.copy_(pm)
        if pc is not None and pc.data_ptr() != comp.data_ptr():
            comp.copy_(pc.to(comp.dtype))
        elif pc is None and comp.data_ptr() != master.data_ptr():
            comp.copy_(master.to(comp.dtype))
        env[(n.id, 0)] = comp if comp.is_contiguous() else comp.contiguous()

    def _ring(self, n: Node):
        """The K / V ring of a context-parallel attention node (transform.cc stamps `cp_levels` on "seq" candidates), or None."""
        lv = [int(l) for l, num in zip(n.attrs.get("cp_levels", []), n.attrs.get("cp_nums", [])) if int(num) > 1]
        if not lv or self.collective is None or self.collective.mesh.world == 1:
            return None
        if len(lv) > 1:
            raise NotImplementedError("context parallelism over more than one mesh level (split the sequence on ONE level)")
        key = tuple(lv)
        if key not in self._rings:
            from ..parallel.ring_attention import RingAttention
            mesh = self.collective.mesh
            self._rings[key] = RingAttention(mesh.group(lv[0]), mesh.group_ranks(lv[0]), mesh.index_in_group(lv[0]),
                                             dry=self.collective.dry)
        return self._rings[key]

    def _bn_sync_levels(self, n: Node) -> List[Tuple[int, int]]:
        """(level, num) pairs over which a batch-split BatchNorm has to complete its statistics: the levels the transform
        recorded, minus time-multiplexed ones (micro-batches of a pipeline normalise on their own, as in the reference)."""
        if self.collective is None or self.collective.mesh.world == 1:
            return []
        out = []
        for lvl, num in zip(n.attrs.get("sync_levels", []), n.attrs.get("sync_nums", [])):
            if int(num) > 1 and self.collective.mesh.group(int(lvl)) is not None:
                out.append((int(lvl), int(num)))
        return out

    def _batchnorm_synced(self, n: Node, ins: List[torch.Tensor]) -> List[torch.Tensor]:
        """Training-mode BatchNorm whose batch is split over devices: per-channel sums are completed across the splitting levels
        (two small all-reduces forward -- mean, then centred second moment, i.e. the same two-pass variance as one device --
        and one backward), so the result equals BatchNorm over the global batch.  The reference gets this from XLA's SPMD
        treatment of the batch reductions; without it data-parallel conv nets silently train with per-shard statistics.
        dgamma / dbeta stay LOCAL partial sums: the plan reduces them with the other gradients."""
        import torch.distributed as dist
        levels = self._bn_sync_levels(n)
        mesh = self.collective.mesh

        def allsum(t: torch.Tensor) -> torch.Tensor:
            if not self.collective.dry:
                for lvl, _ in levels:
                    dist.all_reduce(t, group=mesh.group(lvl))
            return t
        a = n.attrs
        if n.op == "batchnorm":
            xx, gm, bt = ins
        else:
            dy, xx, gm = ins
        if ops.bn_native_ok(xx) and os.environ.get("TEPDIST_BN_SYNC", "native") == "native":
            # native split phases: local sums kernel -> all-reduce of 2 x C floats -> apply kernel with the global count
            shards = 1
            for _, num in levels:
                shards *= num
            key = (self._tag, n.inputs[0 if n.op == "batchnorm" else 1].key())
            if n.op == "batchnorm":
                y, mean, rstd = ops.batchnorm_fwd_synced(xx, gm.float(), bt.float(), a["eps"], allsum, shards, relu=bool(a.get("relu")))
                self.bn_sync_stats[key] = (mean, rstd)
                return [y]
            st_ = self.bn_sync_stats.pop(key, None)
            if st_ is not None:
                mean, rstd = st_
                dx, dgl, dbl = ops.batchnorm_bwd_synced(dy, xx, gm.float(), mean, rstd, allsum, shards)
                dg = self._grad_out(n, 1, n.outputs[1].shape); dg.add_(dgl)
                db = self._grad_out(n, 2, n.outputs[2].shape); db.add_(dbl)
                return [dx, dg, db]
        xf = xx.float()
        cnt = float(xf.numel() // xf.shape[1])
        for _, num in levels:
            cnt *= num
        key = (self._tag, n.inputs[0 if n.op == "batchnorm" else 1].key())
        st_ = self.bn_sync_stats.pop(key, None) if n.op == "batchnorm_bwd" else None
        if st_ is None:
            mean = allsum(xf.sum((0, 2, 3))) / cnt
            var = allsum(((xf - mean.view(1, -1, 1, 1)) ** 2).sum((0, 2, 3))) / cnt
            rstd = torch.rsqrt(var + a["eps"])
        else:
            mean, rstd = st_
        xh = (xf - mean.view(1, -1, 1, 1)) * rstd.view(1, -1, 1, 1)
        if n.op == "batchnorm":
            self.bn_sync_stats[key] = (mean, rstd)      # consumed by the matching batchnorm_bwd
            return [(xh * gm.float().view(1, -1, 1, 1) + bt.float().view(1, -1, 1, 1)).to(xx.dtype)]
        dyf = dy.float()
        g_ = dyf * gm.float().view(1, -1, 1, 1)
        s = allsum(torch.stack([g_.sum((0, 2, 3)), (g_ * xh).sum((0, 2, 3))])) / cnt
        dx = rstd.view(1, -1, 1, 1) * (g_ - s[0].view(1, -1, 1, 1) - xh * s[1].view(1, -1, 1, 1))
        dg = self._grad_out(n, 1, n.outputs[1].shape); dg.add_((dyf * xh).sum((0, 2, 3)))
        db = self._grad_out(n, 2, n.outputs[2].shape); db.add_(dyf.sum((0, 2, 3)))
        return [dx.to(xx.dtype), dg, db]

    def _fused_apply(self) -> None:
        st, o = self.store, self.opt
        kind = o.get("kind")
        if kind == "adamw":
            ops.adamw_step(st.master, st.grad, st.m, st.v, st.compute, st.n_decay, self._lr(1e-3), o.get("beta1", 0.9),
                           o.get("beta2", 0.999), o.get("eps", 1e-8), o.get("weight_decay", 0.0), self.step_count,
                           hyper=self.hyper)
        elif kind == "sgd":
            ops.sgd_step(st.master, st.grad, st.compute, self._lr(1e-2))

    @staticmethod
    def _find_moe_einsums(g: Graph) -> Dict[int, Tuple[str, int]]:
        """einsum node id -> (kind, id of the moe_dispatch_mask node whose route tables it can use).  Matches the GShard
        formulation of models/gpt_moe.py: dispatch "GSEC,GSM->EGCM" / combine "GSEC,EGCM->GSM" with the mask as operand 0
        (which also covers the two gradient einsums that take the mask), and the two d-mask einsums "EGCM,GSM->GSEC" /
        "GSM,EGCM->GSEC", tied to their forward einsum through the op group."""
        found: Dict[int, Tuple[str, int]] = {}
        by_group: Dict[Tuple[int, str], int] = {}
        for n in g.nodes:
            if n.op != "einsum" or len(n.inputs) != 2:
                continue
            eq = str(n.attrs.get("eq", "")).replace(" ", "")
            src = g.nodes[n.inputs[0].node]
            if src.op == "moe_dispatch_mask" and eq in ("GSEC,GSM->EGCM", "GSEC,EGCM->GSM"):
                found[n.id] = ("gather" if eq.endswith("EGCM") else "combine", src.id)
                if not n.backward:
                    by_group[(n.group, eq)] = src.id
        for n in g.nodes:
            if n.op != "einsum" or not n.backward or n.id in found:
                continue
            eq = str(n.attrs.get("eq", "")).replace(" ", "")
            if eq == "EGCM,GSM->GSEC" and (n.group, "GSEC,GSM->EGCM") in by_group:
                found[n.id] = ("dots_eg_first", by_group[(n.group, "GSEC,GSM->EGCM")])
            elif eq == "GSM,EGCM->GSEC" and (n.group, "GSEC,EGCM->GSM") in by_group:
                found[n.id] = ("dots", by_group[(n.group, "GSEC,EGCM->GSM")])
        return found

    @staticmethod
    def find_tp_chains(g: Graph, skip: Optional[set] = None) -> Dict[int, Dict[str, Any]]:
        """LIN (linear / linear_dgrad, no fused epilogue) -> all_reduce(sum) [-> add(bias [N])] [-> add(residual)] chains in
        which every link has exactly one user: {LIN id: {ar, M, N, level, num, bias key, res key, chain node ids}}."""
        users = g.users()
        skip = skip or set()

        def sole_user(nid: int):
            us = users.get((nid, 0), [])
            return g.nodes[us[0][0]] if len(us) == 1 else None

        found: Dict[int, Dict[str, Any]] = {}
        for ar in g.nodes:
            if ar.op != "all_reduce" or int(ar.attrs.get("reduce", 0)) != 0:
                continue
            lin = g.nodes[ar.inputs[0].node]
            if lin.op not in ("linear", "linear_dgrad") or len(lin.inputs) != 2 or sole_user(lin.id) is not ar or lin.id in skip:
                continue
            num, lvl = int(ar.attrs["num"]), int(ar.attrs["level"])
            shp = tuple(lin.outputs[0].shape)
            N = shp[-1]
            M = 1
            for d in shp[:-1]:
                M *= d
            if num < 2 or num > 8 or lin.outputs[0].dtype != "bf16" or N % 8 or M % (128 * num):
                continue
            info: Dict[str, Any] = {"ar": ar.id, "M": M, "N": N, "level": lvl, "num": num, "bias": None, "res": None,
                                    "chain": [ar.id]}
            nxt = sole_user(ar.id)
            if nxt is not None and nxt.op == "add" and len(nxt.inputs) == 2:
                other = nxt.inputs[1] if nxt.inputs[0].node == ar.id else nxt.inputs[0]
                if tuple(g.type_of(other).shape) == (N,):
                    info["bias"] = other.key()
                    info["chain"].append(nxt.id)
                    nn = sole_user(nxt.id)
                    if nn is not None and nn.op == "add" and len(nn.inputs) == 2:
                        o2 = nn.inputs[1] if nn.inputs[0].node == nxt.id else nn.inputs[0]
                        if tuple(g.type_of(o2).shape) == shp and g.type_of(o2).dtype == "bf16":
                            info["res"] = o2.key()
                            info["chain"].append(nn.id)
            found[lin.id] = info
        return found

    def _plan_tp_fusion(self) -> None:
        """Execute every chain found by find_tp_chains as ONE GemmAllReduce call at LIN; the downstream nodes of the chain
        alias its result."""
        if self.dry_comm:
            return
        mesh = self.collective.mesh
        self.tp_fuse = self.find_tp_chains(self.g, set(self.gelu_dual) | set(self.gelu_bwd_fuse) | set(self.alias_of))
        if not self.tp_fuse:
            return
        if TP_FUSED_IMPL is not None:
            GemmAllReduce, SymmBarrier = TP_FUSED_IMPL, (lambda pg: None)
        else:
            from ..parallel.symm import GemmAllReduce, GemmAllReduceMC, McContext, SymmBarrier, symm_backend
        self._tp_ops: Dict[Tuple[int, int, int], Any] = {}
        bar: Dict[int, Any] = {}
        for lid, info in list(self.tp_fuse.items()):
            key = (info["level"], info["M"], info["N"])
            if TP_FUSED_IMPL is None and key not in self._tp_ops:
                # without a multicast-bound group (no NVSwitch multicast / IPC fallback) the chain stays on NCCL: the unicast slot
                # variant (GemmAllReduce) is kept for experiments only (TEPDIST_TP_UNICAST=1), it has not beaten NCCL + cuBLAS
                pg0 = mesh.group(info["level"])
                mc_ok = (os.environ.get("TEPDIST_TP_MC", "1") == "1" and symm_backend(pg0) == "vmm"
                         and (info["M"] * info["N"]) % (8 * info["num"]) == 0)
                if not mc_ok and os.environ.get("TEPDIST_TP_UNICAST", "0") != "1":
                    del self.tp_fuse[lid]
                    continue
            if key not in self._tp_ops:
                pg = mesh.group(info["level"])
                # NVLS (multicast) version when the group's symmetric memory is multicast-bound; unicast slots otherwise
                use_mc = (TP_FUSED_IMPL is None and os.environ.get("TEPDIST_TP_MC", "1") == "1" and symm_backend(pg) == "vmm"
                          and (info["M"] * info["N"]) % (8 * info["num"]) == 0)
                if info["level"] not in bar:
                    bar[info["level"]] = McContext(pg) if use_mc else SymmBarrier(pg)
                if use_mc:
                    self._tp_ops[key] = GemmAllReduceMC(info["M"], info["N"], pg, bar[info["level"]])
                else:
                    self._tp_ops[key] = GemmAllReduce(info["M"], info["N"], pg, bar[info["level"]])
            info["op"] = self._tp_ops[key]
            info["out"] = info["op"].new_output()        # symmetric [M, N] bf16, written by every rank
            # each chain node aliases its immediate predecessor (lin -> ar -> +bias -> +res): that is the dataflow the
            # liveness pass saw, so every key is still in the environment when the next link looks it up
            prev = lid
            for nid in info["chain"]:
                self.alias_of[nid] = (prev, 0)
                prev = nid

    def _run_tp_fused(self, n: Node, ins: List[torch.Tensor]) -> List[torch.Tensor]:
        info = self.tp_fuse[n.id]
        x, w = ins
        x2 = x.reshape(-1, x.shape[-1])
        bias = res = None
        if info["bias"] is not None:
            bias = self._env[info["bias"]]
            if bias.dtype != torch.float32:
                bias = bias.float()
        if info["res"] is not None:
            res = self._env[info["res"]].reshape(info["M"], info["N"]).contiguous()
        y = info["op"](x2.contiguous(), w, info["out"], bias=bias, residual=res, b_mn=(n.op == "linear_dgrad"))
        return [y.view(tuple(n.outputs[0].shape))]

    def _plan_store_init(self) -> None:
        """Gradient slots whose only writer is a weight-gradient GEMM can be written with plain stores (beta = 0) and need
        no zero-fill; everything else (bias / LayerNorm / embedding gradients: accumulating kernels) is zero-filled as
        contiguous ranges of the flat gradient buffer."""
        self._store_init: set = set()
        self._zero_ranges: Optional[List[Tuple[int, int]]] = None
        if not WGRAD_PLAIN_STORE or self.grad_accumulate or not self.store.master.is_cuda:
            return
        st = self.store
        self_init_params = set()
        for (nid, idx), pid in self.grad_binding.items():
            n = self.g.nodes[nid]
            shp = n.outputs[0].shape
            if (n.op == "linear_wgrad" and idx == 0 and n.id not in self.alias_of and len(shp) == 2
                    and ops.wgrad_prefers_store(shp[0], shp[1])):
                self._store_init.add((nid, idx))
                self_init_params.add(pid)
        for n in self.g.nodes:   # unbound weight gradients (general path) are fresh tensors anyway
            shp = n.outputs[0].shape if n.outputs else ()
            if (n.op == "linear_wgrad" and (n.id, 0) not in self.grad_binding and len(shp) == 2
                    and ops.wgrad_prefers_store(shp[0], shp[1])):
                self._store_init.add((n.id, 0))
        ranges: List[Tuple[int, int]] = []
        cur = 0
        for pid in st.order:
            if pid in self_init_params:
                n_el = 1
                for d in st.shape[pid]:
                    n_el *= d
                if st.offset[pid] > cur:
                    ranges.append((cur, st.offset[pid]))
                cur = st.offset[pid] + n_el
        if cur < st.grad.numel():
            ranges.append((cur, st.grad.numel()))
        self._zero_ranges = ranges

    def _zero_grads(self) -> None:
        zr = getattr(self, "_zero_ranges", None)
        if zr is None:
            self.store.grad.zero_()
            return
        for a, b in zr:
            self.store.grad[a:b].zero_()

    # ------------------------------------------------------------------ node dispatch
    def _grad_out(self, n: Node, idx: int, shape) -> torch.Tensor:
        pid = self.grad_binding.get((n.id, idx))
        if pid is not None:
            return self.store.grad_view(pid)
        return torch.zeros(shape, dtype=torch.float32, device=self.device)

    def _exec(self, n: Node, ins: List[torch.Tensor], feeds: Dict[str, torch.Tensor]) -> List[torch.Tensor]:
        op, a = n.op, n.attrs
        dev = self.device
        if op == "parameter":
            return [self.store.compute_view(n.id)]
        if op == "state":
            return [self.store.state[n.id]]
        if op == "boundary":
            raise RuntimeError("boundary values are filled by pipeline Recv tasks")
        if op == "input":
            t = feeds[n.name]
            if t.device != dev:
                t = t.to(dev, non_blocking=True)
            if t.is_floating_point():          # a float batch fed in another precision than the plan declares (fp32 loader, bf16 model)
                wdt = torch_dtype(n.outputs[0].dtype, dev)
                if wdt.is_floating_point and t.dtype != wdt:
                    t = t.to(wdt)
            want = tuple(n.outputs[0].shape)
            if tuple(t.shape) != want:
                full = tuple(a.get("full_shape", want))
                world = self.collective.mesh.world if self.collective is not None else 1
                if tuple(t.shape) == full:      # fed the global batch: take this rank's shard
                    t = shard_of(t, a, self.coords).contiguous()
                elif (want == full and world > 1 and t.dim() >= 1 and t.shape[0] * world == full[0]
                      and tuple(t.shape[1:]) == full[1:]):
                    # the plan keeps this input replicated but every rank fed only its own batch shard (the usual
                    # data-loader contract): assemble the global batch in rank order
                    t = self.collective.gather_input(t)
                else:
                    raise ValueError(f"input '{n.name}': fed shape {tuple(t.shape)}, expected this rank's shard {want} "
                                     f"or the global tensor {full}")
            return [t]
        if op == "constant":
            return [torch.full(n.outputs[0].shape, a["value"], dtype=torch_dtype(n.outputs[0].dtype, dev), device=dev)]
        if op == "embedding":
            return [ops.embedding_fwd(ins[0], ins[1], ins[2])]
        if op == "embedding_bwd":
            dwte = self._grad_out(n, 0, n.outputs[0].shape)
            dwpe = self._grad_out(n, 1, n.outputs[1].shape)
            ops.embedding_bwd(ins[0], ins[1], dwte, dwpe)
            return [dwte, dwpe]
        if op == "layernorm":
            y, mean, rstd = ops.layernorm_fwd(ins[0].contiguous(), ins[1], ins[2], a.get("eps", 1e-5))
            self.ln_stats[(self._tag, n.inputs[0].key(), n.inputs[1].key())] = (mean, rstd)
            return [y]
        if op == "layernorm_bwd":
            key = (self._tag, n.inputs[1].key(), n.inputs[2].key())
            if key in self.ln_stats:
                mean, rstd = self.ln_stats.pop(key)
            else:
                _, mean, rstd = ops.layernorm_fwd(ins[1].contiguous(), ins[2], torch.zeros_like(ins[2]), a.get("eps", 1e-5))
            dg = self._grad_out(n, 1, n.outputs[1].shape)
            db = self._grad_out(n, 2, n.outputs[2].shape)
            dres = None
            if n.id in self.ln_fuse and getattr(self, "_env", None) is not None:
                dres = self._env.get(self.ln_fuse[n.id])
            dx = ops.layernorm_bwd(ins[0], ins[1], ins[2], mean, rstd, dg, db, dres)
            return [dx, dg, db]
        if op in ("linear", "linear_dgrad") and n.id in self.tp_fuse:
            return self._run_tp_fused(n, ins)
        if op == "linear":
            x, w = ins[0], ins[1]
            k = 2
            bias = res = None
            if a.get("bias"):
                bias = ins[k]; k += 1
            if a.get("residual"):
                res = ins[k]
            x2 = x.reshape(-1, x.shape[-1])
            if n.id in self.gelu_dual:
                pre = torch.empty(x2.shape[0], w.shape[0], dtype=x.dtype, device=dev)
                act = torch.empty_like(pre)
                ops.gemm(x2, w, bias=bias, act="gelu", out=pre, out2=act)
                shp = (*x.shape[:-1], w.shape[0])
                return [pre.view(shp), act.view(shp)]
            y = ops.gemm(x2, w, bias=bias, residual=None if res is None else res.reshape(-1, w.shape[0]),
                         out_dtype=x.dtype)
            return [y.view(*x.shape[:-1], w.shape[0])]
        if op == "linear_dgrad":
            dy, w = ins
            dy2 = dy.reshape(-1, dy.shape[-1])
            if n.id in self.gelu_bwd_fuse:
                f = self._env[self.gelu_bwd_fuse[n.id]]
                dx = ops.gemm(dy2, w, b_mn=True, out_dtype=dy.dtype, act="gelu_bwd", aux=f.reshape(-1, w.shape[1]).contiguous())
            else:
                dx = ops.gemm(dy2, w, b_mn=True, out_dtype=dy.dtype)
            return [dx.view(*dy.shape[:-1], w.shape[1])]
        if op == "linear_wgrad":
            dy, x = ins
            acc = self.grad_accumulate or (n.id, 0) not in self._store_init
            if not acc and (n.id, 0) not in self.grad_binding:
                out = torch.empty(n.outputs[0].shape, dtype=torch.float32, device=dev)
            else:
                out = self._grad_out(n, 0, n.outputs[0].shape)
            # sole producer of this gradient in a step without micro-batch accumulation: plain fp32 stores (beta = 0),
            # no atomics and no zero-fill of the slot beforehand
            ops.gemm(dy.reshape(-1, dy.shape[-1]), x.reshape(-1, x.shape[-1]), a_mn=True, b_mn=True, out=out, accumulate=acc,
                     split_k=0 if acc else 1)
            return [out]
        if op == "colsum":
            out = self._grad_out(n, 0, n.outputs[0].shape)
            ops.colsum_acc(ins[0], out)
            return [out]
        if op == "gelu":
            return [ops.gelu_fwd(ins[0].contiguous())]
        if op == "gelu_bwd":
            return [ops.gelu_bwd(ins[0], ins[1])]
        if op == "attention":
            qkv = ins[0]
            seg = ins[1] if len(ins) > 1 else None     # document ids: whole along the sequence (rules.cc AttentionRule)
            B, S, C3 = qkv.shape
            H = a["heads"]
            D = C3 // 3 // H
            q5 = qkv.view(B, S, H, 3, D)  # heads-major: a last-dim split is a split over heads
            ring = self._ring(n)
            if ring is not None:    # context parallel: S is this rank's block of the sequence, K / V blocks ride the ring
                o, lse = ring.forward(q5[:, :, :, 0], q5[:, :, :, 1], q5[:, :, :, 2], causal=a.get("causal", True), segments=seg)
                return [o.reshape(B, S, H * D), lse]
            o, lse = ops.attention_fwd(q5[:, :, :, 0], q5[:, :, :, 1], q5[:, :, :, 2], causal=a.get("causal", True),
                                       seg_q=seg, seg_k=seg)
            return [o.view(B, S, H * D), lse]
        if op == "attention_bwd":
            do, qkv, o, lse = ins[:4]
            seg = ins[4] if len(ins) > 4 else None
            B, S, C3 = qkv.shape
            H = a["heads"]
            D = C3 // 3 // H
            q5 = qkv.view(B, S, H, 3, D)
            dqkv = torch.empty(B, S, H, 3, D, dtype=qkv.dtype, device=dev)
            ring = self._ring(n)
            if ring is not None:
                ring.backward(do.reshape(B, S, H, D), q5[:, :, :, 0], q5[:, :, :, 1], q5[:, :, :, 2], o.reshape(B, S, H, D), lse,
                              causal=a.get("causal", True), dqkv_out=dqkv, segments=seg)
                return [dqkv.view(B, S, C3)]
            ops.attention_bwd(do.reshape(B, S, H, D), q5[:, :, :, 0], q5[:, :, :, 1], q5[:, :, :, 2], o.reshape(B, S, H, D),
                              lse, causal=a.get("causal", True), dqkv_out=dqkv, seg_q=seg, seg_k=seg)
            return [dqkv.view(B, S, C3)]
        if op == "softmax_xent":
            logits, labels = ins
            Vp = logits.shape[-1]
            l2 = logits.reshape(-1, Vp)
            T = int(a.get("global_tokens", l2.shape[0]))  # batch-sharded: partial sum of the GLOBAL mean
            total, _rows = ops.xent_fwd_bwd(l2, labels.reshape(-1), a.get("vocab", Vp), 1.0 / T)
            return [total.reshape(()), l2.view(logits.shape)]
        outs = self._exec_generic(n, ins)
        # mixed-precision operands (bf16 activation + fp32 bias / statistic) promote in torch; the plan's declared element type
        # is what every consumer -- and every hand-written kernel behind it -- expects
        for i, t in enumerate(outs):
            if i < len(n.outputs) and torch.is_tensor(t) and t.is_floating_point():
                want = torch_dtype(n.outputs[i].dtype, dev)
                if want.is_floating_point and t.dtype != want:
                    outs[i] = t.to(want)
        return outs

    def _exec_generic(self, n: Node, ins: List[torch.Tensor]) -> List[torch.Tensor]:
        """HLO-like ops: plain torch math (not on the GPT-2 hot path; conv/bn go through cuDNN exactly as the
        reference's kConvolution custom-calls do, SURVEY K9)."""
        op, a = n.op, n.attrs
        F = torch.nn.functional
        x = ins[0] if ins else None
        if op in ("add", "relu", "relu_bwd") and x.is_cuda:      # own vectorised kernels for the conv-net elementwise ops
            y = ops.ew_native(op, ins[0], ins[1] if len(ins) > 1 else None)
            if y is not None:
                return [y]
        if op == "add": return [ins[0] + ins[1]]
        if op == "sub": return [ins[0] - ins[1]]
        if op == "mul": return [ins[0] * ins[1]]
        if op == "div": return [ins[0] / ins[1]]
        if op == "neg": return [-x]
        if op == "exp": return [x.exp()]
        if op == "log": return [x.log()]
        if op == "tanh": return [x.tanh()]
        if op == "relu": return [x.relu()]
        if op == "relu_bwd": return [ins[0] * (ins[1] > 0).to(ins[0].dtype)]
        if op == "tanh_bwd": return [ins[0] * (1 - ins[1] * ins[1])]
        if op == "scale": return [x * a["alpha"]]
        if op == "sqrt": return [x.sqrt()]
        if op == "rsqrt": return [x.rsqrt()]
        if op == "sigmoid": return [x.sigmoid()]
        if op == "sigmoid_bwd": return [ins[0] * ins[1] * (1 - ins[1])]
        if op == "abs": return [x.abs()]
        if op == "sign": return [x.sign()]
        if op == "maximum": return [torch.maximum(ins[0], ins[1])]
        if op == "minimum": return [torch.minimum(ins[0], ins[1])]
        if op == "compare":
            fn = {"gt": torch.gt, "ge": torch.ge, "lt": torch.lt, "le": torch.le, "eq": torch.eq, "ne": torch.ne}[a.get("direction", "gt")]
            return [fn(ins[0], ins[1])]
        if op == "select": return [torch.where(ins[0].bool(), ins[1], ins[2])]
        if op == "clamp": return [torch.minimum(torch.maximum(ins[1], ins[0]), ins[2])]
        if op == "reverse": return [torch.flip(x, list(a["dims"]))]
        if op == "sort": return [torch.sort(x, dim=int(a["axis"]), descending=bool(a.get("descending", False))).values]
        if op == "iota":
            shp = tuple(n.outputs[0].shape)
            d = int(a.get("dim", 0))
            view = [1] * len(shp)
            view[d] = shp[d]
            r = torch.arange(shp[d], device=self.device, dtype=torch_dtype(n.outputs[0].dtype, self.device))
            return [r.view(view).expand(shp).contiguous()]
        if op == "pad":
            lo, hi = list(a["low"]), list(a["high"])
            spec = []
            for l, h in zip(reversed(lo), reversed(hi)):
                spec += [int(l), int(h)]
            return [F.pad(x, spec, value=float(a.get("value", 0.0)))]
        if op in ("reduce_window", "select_and_scatter"):
            # window reduction over the dims with window > 1 (max or sum); backward re-runs it under autograd on the saved input
            def fwd(t):
                y = t
                for d, (w, st) in enumerate(zip(a["window"], a["strides"])):
                    if w == 1 and st == 1:
                        continue
                    u = y.unfold(d, int(w), int(st))
                    y = u.amax(-1) if a.get("kind", "max") == "max" else u.sum(-1)
                return y
            if op == "reduce_window":
                return [fwd(x.float()).to(x.dtype)]
            xin = ins[0].detach().float().requires_grad_(True)
            with torch.enable_grad():
                y = fwd(xin)
            (gx,) = torch.autograd.grad(y, xin, ins[1].float().reshape(y.shape))
            return [gx.to(ins[0].dtype)]
        if op == "cast": return [x.to(torch_dtype(a["dtype"], self.device))]
        if op == "softmax": return [torch.softmax(x.float(), a["axis"]).to(x.dtype)]
        if op == "softmax_bwd":
            dy, y = ins[0].float(), ins[1].float()
            return [((dy - (dy * y).sum(a["axis"], keepdim=True)) * y).to(ins[0].dtype)]
        if op in ("reduce_sum", "reduce_mean", "reduce_max"):
            axes = tuple(a["axes"])
            if op == "reduce_sum": r = x.float().sum(axes, keepdim=a.get("keepdims", False))
            elif op == "reduce_mean":
                if "mean_divisor" in a: r = x.float().sum(axes, keepdim=a.get("keepdims", False)) / float(a["mean_divisor"])
                else: r = x.float().mean(axes, keepdim=a.get("keepdims", False))
            else: r = x.float().amax(axes, keepdim=a.get("keepdims", False))
            return [r.to(torch_dtype(n.outputs[0].dtype, self.device))]
        if op == "reshape": return [x.reshape(n.outputs[0].shape)]
        if op == "transpose": return [x.permute(a["perm"])]
        if op == "broadcast":
            shape, dims = a["shape"], a["dims"]
            view = [1] * len(shape)
            for i, d in enumerate(dims):
                view[d] = x.shape[i]
            return [x.reshape(view).expand(shape)]
        if op == "slice":
            idx = tuple(slice(s, l) for s, l in zip(a["starts"], a["limits"]))
            return [x[idx]]
        if op == "pad_zero":
            out = torch.zeros(a["shape"], dtype=x.dtype, device=x.device)
            idx = tuple(slice(s, s + d) for s, d in zip(a["starts"], x.shape))
            out[idx] = x
            return [out]
        if op == "concat": return [torch.cat(ins, a["axis"])]
        if op == "gather": return [ins[0][ins[1].long()]]
        if op == "scatter_add":
            idx, dy = ins
            out = self._grad_out(n, 0, n.outputs[0].shape)
            out.index_add_(0, idx.reshape(-1).long(), dy.reshape(-1, dy.shape[-1]).float())
            return [out]
        if op in ("moe_dispatch_mask", "moe_dispatch_mask_bwd"):
            gates = (ins[0] if op == "moe_dispatch_mask" else ins[1]).float()
            C, k = int(a["capacity"]), int(a.get("top_k", 2))
            Gn, Sn, E = gates.shape
            remaining = gates.clone()
            offset = torch.zeros(Gn, 1, E, device=gates.device)
            sel = torch.zeros(Gn, Sn, E, C, device=gates.device)   # 0/1 slot assignment
            r_e, r_c, r_w = [], [], []
            for _ in range(k):
                idx = remaining.argmax(-1)
                mask = F.one_hot(idx, E).float()
                pos = (mask.cumsum(1) - 1 + offset) * mask
                keep = (pos < C).float() * mask
                sel = sel + keep.unsqueeze(-1) * F.one_hot(pos.long().clamp(max=C - 1), C).float()
                if op == "moe_dispatch_mask" and MOE_SPARSE:
                    kept = keep.sum(-1) > 0                                   # [G, S]: this choice got a slot
                    r_e.append(torch.where(kept, idx, torch.full_like(idx, -1)).int())
                    r_c.append((pos * mask).sum(-1).long().clamp(max=C - 1).int())
                    r_w.append(gates.gather(-1, idx.unsqueeze(-1)).squeeze(-1) * kept)
                offset = offset + mask.sum(1, keepdim=True)
                remaining = remaining.masked_fill(mask.bool(), float("-inf"))
            if op == "moe_dispatch_mask":
                out = (gates.unsqueeze(-1) * sel).to(torch_dtype(n.outputs[0].dtype, self.device))
                if MOE_SPARSE:
                    # route tables of this mask (token -> its <= k slots; slot -> its one token), kept for the dispatch /
                    # combine einsums that consume the mask and for the gradient einsums that produce d mask
                    re_, rc_, gw_ = torch.stack(r_e, -1).contiguous(), torch.stack(r_c, -1).contiguous(), torch.stack(r_w, -1).contiguous()
                    slot_src = torch.full((Gn, E * C), -1, dtype=torch.int32, device=gates.device)
                    slot_w = torch.zeros(Gn, E * C, dtype=torch.float32, device=gates.device)
                    s_idx = torch.arange(Sn, device=gates.device, dtype=torch.int32).view(1, Sn, 1).expand(Gn, Sn, k)
                    flat = (re_.clamp(min=0).long() * C + rc_.long())
                    flat = torch.where(re_ >= 0, flat, torch.full_like(flat, E * C))          # dropped routes -> a dummy column
                    pad_src = torch.cat([slot_src, slot_src.new_full((Gn, 1), -1)], 1)
                    pad_w = torch.cat([slot_w, slot_w.new_zeros(Gn, 1)], 1)
                    pad_src.scatter_(1, flat.reshape(Gn, -1), s_idx.reshape(Gn, -1))
                    pad_w.scatter_(1, flat.reshape(Gn, -1), gw_.reshape(Gn, -1).float())
                    self._moe_routes[(self._tag, n.id)] = {"re": re_, "rc": rc_, "gw": gw_.float().contiguous(), "E": E, "C": C,
                                                           "slot_src": pad_src[:, :E * C].reshape(Gn, E, C).contiguous(),
                                                           "slot_w": pad_w[:, :E * C].reshape(Gn, E, C).contiguous()}
                return [out]
            return [(ins[0].float() * sel).sum(-1).to(ins[1].dtype)]
        if op == "one_hot":
            return [F.one_hot(x.long(), a["depth"]).to(torch_dtype(n.outputs[0].dtype, self.device))]
        if op == "matmul":
            A, B = ins
            ta, tb = a["ta"], a["tb"]
            if (A.is_cuda and A.dtype == torch.bfloat16 and A.dim() == B.dim() and A.dim() in (2, 3)
                    and A.is_contiguous() and B.is_contiguous() and all(d % 8 == 0 for d in A.shape[-2:] + B.shape[-2:])):
                # logical A is (M,K): stored [M,K] (ta=False) or [K,M] (ta=True, i.e. MN-major); same for B
                return [ops.gemm(A, B, a_mn=ta, b_mn=not tb)]
            if ta: A = A.transpose(-1, -2)
            if tb: B = B.transpose(-1, -2)
            return [torch.matmul(A, B)]
        if op == "einsum" and n.id in self._moe_einsum:
            kind, mask_id = self._moe_einsum[n.id]
            rt = self._moe_routes.get((self._tag, mask_id))
            if rt is not None:
                # the route tables describe the mask AS THIS RANK HOLDS IT ([G_local, S, E, C]); an einsum the planner sharded
                # differently (e.g. a gradient einsum split over E instead of G) sees other local extents: keep it dense
                Gr, Sr, Kr = rt["re"].shape
                Er, Cr = rt["E"], rt["C"]
                tok = ins[0] if kind == "dots" else ins[1]        # the [G, S, M] operand (gather / dots_eg_first) ...
                exp = ins[1] if kind in ("dots", "combine") else ins[0]   # ... and the [E, G, C, M] one
                ok = True
                if kind in ("gather", "dots", "dots_eg_first"):
                    ok &= tok.dim() == 3 and tuple(tok.shape[:2]) == (Gr, Sr)
                if kind in ("combine", "dots", "dots_eg_first"):
                    ok &= exp.dim() == 4 and tuple(exp.shape[:3]) == (Er, Gr, Cr)
                if kind in ("gather", "combine"):
                    ok &= tuple(ins[0].shape) == (Gr, Sr, Er, Cr)
                if not ok:
                    rt = None
            if rt is not None:
                if kind == "gather":         # "GSEC,GSM->EGCM": dispatch / d(expert output) of the combine
                    return [ops.moe_gather_scale(ins[1].contiguous(), rt["slot_src"], rt["slot_w"], rt["E"], rt["C"])]
                if kind == "combine":        # "GSEC,EGCM->GSM": combine / d(tokens) of the dispatch
                    return [ops.moe_combine_sum(ins[1].contiguous(), rt["re"], rt["rc"], rt["gw"], ins[0].shape[1])]
                # d mask: "EGCM,GSM->GSEC" (dots of d dispatched rows with tokens) / "GSM,EGCM->GSEC" (d out with expert outputs)
                a_, b_ = (ins[1], ins[0]) if kind == "dots_eg_first" else (ins[0], ins[1])
                dots = ops.moe_route_dots(a_.contiguous(), b_.contiguous(), rt["re"], rt["rc"])
                Gn, Sn, K_ = dots.shape
                dense = torch.zeros(Gn, Sn, rt["E"] * rt["C"] + 1, dtype=torch.float32, device=dots.device)
                flat = rt["re"].clamp(min=0).long() * rt["C"] + rt["rc"].long()
                flat = torch.where(rt["re"] >= 0, flat, torch.full_like(flat, rt["E"] * rt["C"]))
                dense.scatter_(2, flat, dots)
                return [dense[:, :, :rt["E"] * rt["C"]].reshape(Gn, Sn, rt["E"], rt["C"]).to(torch_dtype(n.outputs[0].dtype, self.device))]
        if op == "einsum":
            # own batched tcgen05 GEMM for bf16 operands on the GPU (expert FFNs, dispatch / combine and their gradients);
            # torch.einsum for the CPU oracle and for patterns outside the kernel's alignment rules
            if (ins[0].is_cuda and ins[0].dtype == torch.bfloat16 and ins[1].dtype == torch.bfloat16
                    and os.environ.get("TEPDIST_EINSUM", "own") != "torch"):
                return [ops.einsum(a["eq"], ins[0], ins[1])]
            return [torch.einsum(a["eq"], ins[0], ins[1])]
        # convolutions: own path = NHWC im2col / col2im kernels + tcgen05 GEMMs (ops/csrc/conv_sm100.cu); cuDNN through torch
        # is the reference-semantics path (TEPDIST_CONV=cudnn) and the CPU oracle
        if op == "conv2d":
            if ops.conv_native_ok(ins[0], ins[1]):
                return [ops.conv2d_fwd(ins[0], ins[1], a["stride"], a["padding"])]
            return [F.conv2d(ins[0], ins[1], stride=a["stride"], padding=a["padding"])]
        if op == "conv2d_dgrad":
            dy, w = ins
            if ops.conv_native_ok(dy, w):
                return [ops.conv2d_dgrad(dy, w, n.outputs[0].shape, a["stride"], a["padding"])]
            return [torch.nn.grad.conv2d_input(n.outputs[0].shape, w, dy, stride=a["stride"], padding=a["padding"])]
        if op == "conv2d_wgrad":
            dy, xx = ins
            if ops.conv_native_ok(xx, dy.new_empty((n.outputs[0].shape[0], 1, 1, 1))):
                gw = ops.conv2d_wgrad(dy, xx, n.outputs[0].shape, a["stride"], a["padding"])
            else:
                gw = torch.nn.grad.conv2d_weight(xx, n.outputs[0].shape, dy, stride=a["stride"], padding=a["padding"])
            out = self._grad_out(n, 0, n.outputs[0].shape)
            out.add_(gw.float())
            return [out]
        if op in ("batchnorm", "batchnorm_bwd") and self._bn_sync_levels(n):
            return self._batchnorm_synced(n, ins)
        if op == "batchnorm":
            xx, gm, bt = ins
            if ops.bn_native_ok(xx) and gm.dtype == torch.float32:
                y, mean, rstd = ops.batchnorm_fwd(xx, gm, bt, a["eps"])
                self.bn_stats[(self._tag, n.inputs[0].key())] = (mean, rstd)     # consumed by the matching batchnorm_bwd
                return [y]
            return [F.batch_norm(xx, None, None, gm.to(xx.dtype), bt.to(xx.dtype), True, 0.0, a["eps"])]
        if op == "batchnorm_bwd":
            dy, xx, gm = ins
            st_ = self.bn_stats.pop((self._tag, n.inputs[1].key()), None)
            if st_ is not None and ops.bn_native_ok(xx) and gm.dtype == torch.float32:
                dx, dgm, dbt = ops.batchnorm_bwd(dy, xx, gm, st_[0], st_[1])
                dg = self._grad_out(n, 1, n.outputs[1].shape); dg.add_(dgm)
                db = self._grad_out(n, 2, n.outputs[2].shape); db.add_(dbt)
                return [dx, dg, db]
            xf, dyf = xx.float(), dy.float()
            mean = xf.mean((0, 2, 3), keepdim=True)
            var = xf.var((0, 2, 3), unbiased=False, keepdim=True)
            rstd = torch.rsqrt(var + a["eps"])
            xh = (xf - mean) * rstd
            g_ = dyf * gm.float().view(1, -1, 1, 1)
            dx = rstd * (g_ - g_.mean((0, 2, 3), keepdim=True) - xh * (g_ * xh).mean((0, 2, 3), keepdim=True))
            dg = self._grad_out(n, 1, n.outputs[1].shape); dg.add_((dyf * xh).sum((0, 2, 3)))
            db = self._grad_out(n, 2, n.outputs[2].shape); db.add_(dyf.sum((0, 2, 3)))
            return [dx.to(xx.dtype), dg, db]
        # pooling: own NHWC kernels on the GPU (conv_sm100.cu; gather-form max-pool backward from the saved input / output instead of
        # re-running the forward under autograd), torch ops on CPU
        if op == "maxpool2d": return [ops.maxpool2d_fwd(x, a["k"], a["stride"], a["padding"])]
        if op == "maxpool2d_bwd": return [ops.maxpool2d_bwd(ins[0], ins[1], ins[2], a["k"], a["stride"], a["padding"])]
        if op == "global_avgpool": return [ops.global_avgpool_fwd(x)]
        if op == "global_avgpool_bwd": return [ops.global_avgpool_bwd(x, tuple(n.outputs[0].shape))]
        if op in ("all_reduce", "all_gather", "reduce_scatter", "all_to_all", "dynamic_slice", "send", "recv"):
            assert self.collective is not None, f"collective op {op} without a communicator"
            # (a bound gradient is ADDED into the flat buffer by the caller: with micro-batching the collective runs once
            #  per micro-batch and must accumulate, so it never writes the buffer in place)
            return self.collective.run(n, ins, None)
        raise NotImplementedError(op)
