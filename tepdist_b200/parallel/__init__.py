"""Parallel execution: plan on rank 0 (the reference's master), dispatch the plan, build per-rank executors."""
from __future__ import annotations

import json
from typing import Any, Dict, Optional

import torch
import torch.distributed as dist

from ..ir import Graph


def plan_spmd(graph: Graph, num: int, strategy: str = "auto", options: Optional[Dict[str, Any]] = None):
    """Run the C++ planner + SPMD transform for one mesh level of `num` devices.
    Returns (sharded ir.Graph, info dict)."""
    from .. import _C
    from ..planner import from_native, merge_client_attrs, to_native
    options = dict(options or {})
    g = graph
    sp = strategy == "tpsp"      # tensor parallel in the sequence-parallel form: reduce-scatter / all-gather around the token-wise ops
    if sp:
        strategy = "tp"
    if strategy in ("dp", "tp", "cp"):
        g = Graph.from_dict(graph.to_dict())
        ids = _document_id_inputs(g.nodes)
        for n in g.nodes:
            if n.op == "input":
                # "cp" (context parallel): every [batch, sequence, ...] sample input is cut along the SEQUENCE, except attention's
                # document ids, which every rank keeps whole (rules.cc AttentionRule)
                dim = {"dp": 0, "tp": -1}.get(strategy, 1 if len(n.outputs[0].shape) >= 2 and n.id not in ids else -1)
                n.attrs["sharding"] = {"0": {"dim": dim, "num": num}}
    cg = to_native(g)
    o = _C.SpmdOptions()
    o.num = num
    if strategy in ("dp", "tp", "cp"):
        o.ignore_annotation = False
    if strategy == "cp":
        o.context_parallel = True
    if sp:
        o.sequence_parallel = True
    if strategy == "tp":
        o.var_mem_limit = 1.0  # force every weight MATRIX to be stored sharded -> tensor parallel (vectors stay whole)
        o.mem_split_min_rank = 2
    from .. import config
    o.hw = config.hw_profile()
    config.check_num_gradients(sum(1 for n in graph.nodes if n.op.startswith("apply_")))
    for k, v in {**config.spmd_overrides(), **options}.items():   # flags (ServiceEnv) < explicit call arguments
        if hasattr(o, k):
            setattr(o, k, v)
    # "dp" / "rule": annotation-driven rule mode (reference FastSpmdStrategy, RULE_MODE=true): the batch split on the
    # sample inputs is propagated through the graph, variables stay replicated, gradients come out partial.
    _C.unknown_ops(True)
    plan = _C.plan_spmd_by_rules(cg, o) if strategy in ("rule", "dp") else _C.plan_spmd_level(cg, o)
    unknown = list(_C.unknown_ops(True))
    if unknown:
        import warnings
        warnings.warn(f"SPMD planner: no sharding rule for op(s) {sorted(unknown)}: they (and what only they connect) stay replicated; "
                      "add a rule to csrc/rules.cc to let the planner shard through them")
    if getattr(plan.stats, "ignored_annotations", 0):
        import warnings
        warnings.warn(f"SPMD planner: {plan.stats.ignored_annotations} sharding annotation(s) cannot be honoured by any strategy of "
                      "their node (dimension not divisible by the device count?) and were ignored")
    if plan.stats.infeasible_subgraphs:
        import warnings
        warnings.warn(f"SPMD planner: {plan.stats.infeasible_subgraphs} sub-graph(s) without a consistent assignment; their nodes keep "
                      "their first candidate (the plan is valid but not optimised there)")
    cg.split_nums = [num]
    cg.share_dev = [False]
    tg, st = _C.spmd_transform(cg, plan, 0, num)
    buckets = _C.combine_gradient_collectives(tg, int(options.get("bucket_bytes", 64 << 20)))
    out = from_native(tg)
    merge_client_attrs(out, graph)
    tags: Dict[str, int] = {}
    heavy = ("linear", "linear_dgrad", "matmul", "einsum", "conv2d", "conv2d_dgrad")
    for i in range(cg.num_nodes()):
        if cg.node_op(i) not in heavy:
            continue
        c = plan.choice[i]
        w_split = any(cg.node_op(src) == "parameter" and not c.ins[k].is_glue() for k, (src, _) in enumerate(cg.node_inputs(i)))
        act_split = any(not s.is_glue() for s in list(c.ins) + list(c.outs))
        kind = "tp" if w_split else ("dp" if act_split else "replicated")
        if cg.node_op(i) == "einsum" and c.tag == "batch" and w_split:
            kind = "ep"   # a batch (expert) dim of the weight is split: expert parallel
        tags[kind] = tags.get(kind, 0) + 1
    ring = sum(1 for i in range(cg.num_nodes()) if cg.node_op(i) == "attention" and plan.choice[i].tag == "seq")
    info = {"context_parallel": ring, "comm_info": st.comm_info(), "comm_bytes": plan.stats.comm_bytes, "solve_seconds": plan.stats.solve_seconds,
            "subgraphs": plan.stats.num_subgraphs, "distinct_subgraphs": plan.stats.distinct_subgraphs,
            "collectives": dict(plan.stats.collectives), "dot_strategies": tags, "grad_buckets": buckets, "infeasible_subgraphs": plan.stats.infeasible_subgraphs,
            "strategies_txt": _C.dump_strategies(cg, plan), "unknown_ops": sorted(unknown)}
    return out, info


def _document_id_inputs(nodes) -> set:
    """Ids of the input nodes that feed attention its document ids (the optional last operand of attention / attention_bwd),
    followed back through single-operand nodes (the slices an earlier mesh level inserted).  `nodes`: ir Nodes, or
    (op, [input node ids]) pairs, indexed by node id."""
    g = [(n.op, [v.node for v in n.inputs]) if hasattr(n, "op") else n for n in nodes]
    out = set()
    for op, ins in g:
        k = {"attention": 1, "attention_bwd": 4}.get(op)
        if k is not None and len(ins) > k:
            i = ins[k]
            while g[i][0] != "input" and len(g[i][1]) == 1:
                i = g[i][1][0]
            out.add(i)
    return out


def plan_spmd_mesh(graph: Graph, nums, kinds):
    """Multi-dimensional SPMD mesh (reference: one split ordinal per mesh dimension, dist_spec.h:130-227): plan and transform
    level 0 over nums[0] devices, then level 1 over nums[1] devices on the already sharded graph, ...  `kinds[i]` is
    "dp" (cost-based, memory unconstrained: batch split wins), "tp" (weights forced sharded) or "auto".
    Returns (sharded ir.Graph, info)."""
    from .. import _C, config
    from ..planner import from_native, merge_client_attrs, to_native
    cg = to_native(graph)
    cg.split_nums = [int(n) for n in nums]
    cg.share_dev = [False] * len(nums)
    colls: Dict[str, int] = {}
    comm = 0.0
    secs = 0.0
    infeasible = 0
    for lvl, (num, kind) in enumerate(zip(nums, kinds)):
        o = _C.SpmdOptions()
        o.num = int(num)
        for k, v in config.spmd_overrides().items():
            if hasattr(o, k):
                setattr(o, k, v)
        if kind in ("tp", "tpsp"):
            o.var_mem_limit = 1.0
            o.mem_split_min_rank = 2
            o.sequence_parallel = kind == "tpsp"
        if kind == "cp":    # sequence split seeded on the sample inputs of THIS level, attention keeps it (K / V ring)
            o.context_parallel = True
            o.ignore_annotation = False
            # ... except attention's document ids: every rank keeps them whole along the sequence (rules.cc AttentionRule)
            ids = _document_id_inputs([(cg.node_op(i), [v[0] for v in cg.node_inputs(i)]) for i in range(cg.num_nodes())])
            for i in range(cg.num_nodes()):
                if cg.node_op(i) == "input":
                    cg.set_node_attr(i, "shard_dim", 1 if len(cg.node_outputs(i)[0][0]) >= 2 and i not in ids else -1)
        plan = _C.plan_spmd_level(cg, o)
        if kind == "cp":
            for i in range(cg.num_nodes()):
                if cg.node_op(i) == "input":
                    cg.erase_node_attr(i, "shard_dim")
        infeasible += plan.stats.infeasible_subgraphs
        cg, _ = _C.spmd_transform(cg, plan, lvl, int(num))
        for k, v in dict(plan.stats.collectives).items():
            colls[k] = colls.get(k, 0) + int(v)
        comm += plan.stats.comm_bytes
        secs += plan.stats.solve_seconds
    out = from_native(cg)
    merge_client_attrs(out, graph)
    if infeasible:
        import warnings
        warnings.warn(f"SPMD planner: {infeasible} sub-graph(s) without a consistent assignment over the mesh levels")
    info = {"collectives": colls, "comm_bytes": comm, "solve_seconds": secs, "mesh": [int(n) for n in nums], "kinds": list(kinds),
            "infeasible_subgraphs": infeasible}
    return out, info


def _parse_mesh_strategy(strategy: str):
    """"dp4tp2" / "tp2dp4" / "dp2tp2dp2" -> ([4, 2], ["dp", "tp"]) ; None when `strategy` is not a mesh spec."""
    import re
    parts = re.findall(r"(dp|tpsp|tp|cp|auto)(\d+)", strategy)
    if len(parts) < 2 or "".join(k + n for k, n in parts) != strategy:
        return None
    # tensor-parallel levels are planned first: the data-parallel level (with its ZeRO-style optimizer sharding) then acts
    # on the already tensor-sharded variables, which is the nesting the executor's in-place sharded update understands
    parts.sort(key=lambda kn: 0 if kn[0] in ("tp", "tpsp") else 1)
    return [int(n) for _, n in parts], [k for k, _ in parts]


def classify_parallelism(info: Dict[str, Any], num: int) -> str:
    if info.get("context_parallel"):
        return f"cp{num}"      # the sequence split runs through attention (K / V ring); everything else is token-wise
    t = info.get("dot_strategies", {})
    if not t:
        return f"replicated{num}"
    kind = max(t, key=t.get)
    c = info.get("collectives", {})
    if kind == "dp" and c.get("reduce_scatter", 0) > c.get("all_reduce", 0):
        return f"dp{num}+zero1"
    return f"{kind}{num}"


def plan_pipeline(graph: Graph, world: int, stages: int, micro: int, options: Optional[Dict[str, Any]] = None):
    """AutoParallel (config or exploration mode) -> (transformed ir.Graph with stages, plan info, per-device task lists)."""
    from .. import _C
    from ..planner import from_native, merge_client_attrs, to_native
    cg = to_native(graph)
    ap = _C.AutoParallelOptions()
    ap.num_devices = world
    if stages > 0:
        ap.mode = "config"
        ap.num_stages, ap.num_micro_batches = stages, micro
    import os
    if os.environ.get("TEPDIST_SPMD_RULE_MODE") == "1":
        ap.spmd_rule_mode = True
    from .. import config
    ap.hw = config.hw_profile()
    config.check_num_gradients(sum(1 for n in graph.nodes if n.op.startswith("apply_")))
    for k, v in {**config.auto_parallel_overrides(), **(options or {})}.items():
        if hasattr(ap, k):
            setattr(ap, k, v)
    plan = _C.auto_parallel(cg, ap)
    pr = plan.proposal
    out = from_native(plan.graph)
    merge_client_attrs(out, graph)
    # task graph + 1F1B schedule (C++ runtime core): the plan is decomposed into its DefContext tree (SyncFreeDecompose: CG /
    # GAINIT / GA / AG; StageDecompose: CG_SLICE_<s>_{F,B}, AG_SLICE_<s> + the neighbour-only transfer list) and the TaskDAG is
    # COMPILED from that tree -- task costs are the contexts' FLOPs, Send / Recv bytes the transfer list (CompileTaskDAG)
    hw = config.hw_profile()
    if config.pp_bandwidth() is not None:
        hw.link_bw = config.pp_bandwidth()
    dec = _C.sync_free_decompose(plan.graph, 0 if pr.micro > 1 else -1)
    xfers = _C.stage_decompose(plan.graph, pr.stages, dec)
    dag, sp = _C.compile_task_dag(plan.graph, dec, xfers, pr.micro, pr.spmd, hw)
    so = _C.ScheduleOptions()
    for k, v in config.schedule_overrides().items():
        setattr(so, k, v)
    sch = _C.schedule_tasks(dag, sp, so)
    def released_micros(t):
        # GC plan of the scheduler (ComputeReleasePlan): the micro-batches whose LAST value on this device -- the output of
        # the backward bundle -- dies after task t; the stage worker drops the whole micro-batch environment there
        return [dag.nodes[r].micro for r in dag.nodes[t].mem_to_release
                if dag.nodes[r].type == _C.TaskType.Output and dag.nodes[r].backward]
    tasks = {int(dev): [{"type": dag.nodes[t].type.name, "micro": dag.nodes[t].micro, "backward": dag.nodes[t].backward,
                         "stage": dag.nodes[t].stage, "name": dag.nodes[t].name, "buffer_id": dag.nodes[t].buffer_id,
                         "buffer_reused": dag.nodes[t].buffer_reused, "release": released_micros(t)} for t in lst]
             for dev, lst in sch.device_tasks.items()}
    info = {"stages": pr.stages, "micro": pr.micro, "spmd": pr.spmd, "log": plan.log, "eval": repr(plan.eval),
            "def_contexts": [c.name for c in dec.ctx], "stage_fwd_seconds": list(sp.fwd_seconds), "stage_bwd_seconds": list(sp.bwd_seconds),
            "boundary_bytes": list(sp.boundary_bytes),
            "makespan_est": sch.makespan, "bubble_est": sch.bubble_ratio, "cut_bytes": plan.stage_plan.cut_bytes,
            "stage_method": plan.stage_plan.method, "candidates": list(plan.candidates)}
    return out, info, tasks


class PipelineRunner:
    """Adapter exposing the Executor-like `step(feeds)` interface for a pipeline stage worker."""

    def __init__(self, worker, tasks, device):
        self.worker, self.tasks, self.device = worker, tasks, device
        self.store = worker.exec.store

    def step(self, feeds):
        from ..runtime.pipeline import run_pipeline_step
        loss = run_pipeline_step(self.worker, self.tasks, feeds)
        t = torch.tensor([loss if loss is not None else 0.0], dtype=torch.float32, device=self.device)
        # the loss lives on the last stage: share it so every rank reports the same number
        import torch.distributed as dist
        dist.broadcast(t, src=dist.get_world_size() - 1)
        return [t.reshape(())]


def build_pipeline(graph: Graph, trainer, stages: int, micro: int, comm_mode: str, seed: int, use_cuda_graph: bool = False):
    from ..runtime.pipeline import StageWorker
    from .collectives import CollectiveRunner
    from .mesh import DeviceMesh
    world, rank = trainer.world, trainer.rank
    payload = [None]
    if rank == 0:
        g2, info, tasks = plan_pipeline(graph, world, stages, micro)
        from ..utils import trace
        trace.log_plan(info, f"pp{info['stages']}x spmd{info['spmd']} micro{info['micro']}")
        if trace.debug_enabled():
            trace.dump_plan_artifacts(g2, info, extra={"local-task-lists.json": json.dumps(tasks, indent=1)})
        payload[0] = json.dumps({"graph": g2.to_dict(), "info": info, "tasks": tasks})
    dist.broadcast_object_list(payload, src=0)
    d = json.loads(payload[0])
    g2 = Graph.from_dict(d["graph"])
    info = d["info"]
    S, M, n = info["stages"], info["micro"], info["spmd"]
    trainer.plan_info.update({k: v for k, v in info.items() if k != "log"})
    trainer.plan_info["parallelism"] = f"pp{S}" + (f"xspmd{n}" if n > 1 else "") + f"/micro{M}"
    levels, shared = [], []
    if M > 1:
        levels.append(M); shared.append(True)
    if n > 1:
        levels.append(n); shared.append(False)
    levels.append(S); shared.append(False)
    stage_level = len(levels) - 1
    layout = [stage_level] + [l for l in range(len(levels)) if l != stage_level]
    mesh = DeviceMesh(levels, shared, layout, rank=rank, world=world)
    mesh.build_process_groups()
    trainer.mesh = mesh
    coords = mesh.coords()
    stage = coords[stage_level]
    for l, sh in enumerate(shared):
        if sh:
            coords[l] = 0
    base = mesh.stride(stage_level)
    worker = StageWorker(g2, stage, S, M, 0 if M > 1 else -1, trainer.device, rank - base if stage > 0 else None,
                         rank + base if stage < S - 1 else None, seed=seed, collective=CollectiveRunner(mesh), coords=coords,
                         comm_mode=comm_mode, use_cuda_graph=use_cuda_graph)
    worker.plan_transfers()
    tasks = d["tasks"][str(stage * n)]
    return PipelineRunner(worker, tasks, trainer.device)


def plan_and_build(graph: Graph, trainer, strategy: str, comm_mode: str, use_cuda_graph: bool, seed: int):
    from ..runtime.executor import Executor
    from .. import config
    strategy = config.resolve_strategy(strategy)
    if strategy == "explore":
        # AutoParallel exploration mode (reference auto_parallel.cc:236-324): every device-mesh proposal (stages x
        # micro-batches x SPMD) is planned and scored by the evaluator; the winner is then built like a configured plan
        payload = [None]
        if trainer.rank == 0:
            _, xinfo, _ = plan_pipeline(graph, trainer.world, 0, 0)
            payload[0] = json.dumps({"stages": xinfo["stages"], "micro": xinfo["micro"], "spmd": xinfo["spmd"]})
        dist.broadcast_object_list(payload, src=0)
        x = json.loads(payload[0])
        trainer.plan_info["explored"] = x
        strategy = f"pp{x['stages']}m{x['micro']}" if x["stages"] > 1 else "auto"
    if strategy.startswith("pp"):   # "pp<S>" or "pp<S>m<M>": config-mode pipeline (NUM_STAGES / NUM_MICRO_BATCHES)
        body = strategy[2:]
        S_, _, M_ = body.partition("m")
        stages = int(S_)
        micro = int(M_) if M_ else max(2, 2 * stages)
        import os
        return build_pipeline(graph, trainer, stages, micro, comm_mode, seed,
                              use_cuda_graph=use_cuda_graph and os.environ.get("TEPDIST_PP_GRAPH", "1") == "1")
    from .collectives import CollectiveRunner
    from .mesh import DeviceMesh
    world, rank = trainer.world, trainer.rank
    mesh_spec = _parse_mesh_strategy(strategy)
    if mesh_spec is not None:      # multi-dimensional SPMD mesh, e.g. "dp4tp2": data parallel over 4 x tensor parallel over 2
        nums, kinds = mesh_spec
        total = 1
        for n_ in nums:
            total *= n_
        assert total == world, f"strategy {strategy} needs {total} devices, world is {world}"
        payload = [None]
        if rank == 0:
            sharded, info = plan_spmd_mesh(graph, nums, kinds)
            from ..utils import trace
            trace.log_plan(info, strategy)
            if trace.debug_enabled():
                trace.dump_plan_artifacts(sharded, info)
            payload[0] = json.dumps({"graph": sharded.to_dict(), "info": info})
        dist.broadcast_object_list(payload, src=0)
        d = json.loads(payload[0])
        sharded = Graph.from_dict(d["graph"])
        trainer.plan_info.update(d["info"])
        trainer.plan_info["parallelism"] = "x".join(f"{k}{n}" for k, n in zip(kinds, nums))
        mesh = DeviceMesh(nums, [False] * len(nums), rank=rank, world=world)
        mesh.build_process_groups()
        trainer.mesh = mesh
        runner = CollectiveRunner(mesh, comm_dtype=config.comm_dtype())
        return Executor(sharded, trainer.device, seed=seed, use_cuda_graph=use_cuda_graph, collective=runner,
                        coords=mesh.coords(), comm_mode=comm_mode)
    payload = [None]
    if rank == 0:
        sharded, info = plan_spmd(graph, world, strategy)
        from ..utils import trace
        trace.log_plan(info, classify_parallelism(info, world))
        if trace.debug_enabled():
            trace.dump_plan_artifacts(sharded, info)
        payload[0] = json.dumps({"graph": sharded.to_dict(), "info": {k: v for k, v in info.items() if k != "strategies_txt"}})
    dist.broadcast_object_list(payload, src=0)   # master -> workers plan dispatch (reference DispatchPlan RPC)
    d = json.loads(payload[0])
    sharded = Graph.from_dict(d["graph"])
    trainer.plan_info.update(d["info"])
    trainer.plan_info["parallelism"] = classify_parallelism(d["info"], world)
    mesh = DeviceMesh([world], [False], rank=rank, world=world)
    mesh.build_process_groups()
    trainer.mesh = mesh
    runner = CollectiveRunner(mesh, comm_dtype=config.comm_dtype())
    return Executor(sharded, trainer.device, seed=seed, use_cuda_graph=use_cuda_graph, collective=runner,
                    coords=mesh.coords(), comm_mode=comm_mode)
