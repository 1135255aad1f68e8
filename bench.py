#!/usr/bin/env python
"""Headline benchmark: GPT-2 345M training throughput (tokens/s, whole job) on N B200s of one node.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (N>1 via torch.distributed.run), one JSON
line from rank 0.  Metric/config = BASELINE.json: GPT-2 (examples/GPT2/345M.json: 24 layers, d=1024,
16 heads, ctx 1024, vocab 50257, batch 4 per model replica, AdamW), bf16 compute / fp32 master+optimizer,
synthetic `fake_input` tokens, random-init weights.  Every step = forward + backward + gradient sync +
optimizer update.  `--impl reference` is the reference arm (see DESIGN.md: the TensorFlow-fork reference
cannot be installed offline, so it reports `unavailable`).

Tokens and initial weights are seeded, so runs with the same arguments start from identical inputs; `--dump-outputs DIR`
writes what the last timed step computed, so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REF_BASELINE_TOKENS_PER_S = None  # BASELINE.md: the reference publishes no number

# the benchmark may run from a read-only tree: leave it as the build left it
sys.dont_write_bytecode = True


def clocks_sampler(stop_evt, samples, gpu_index):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not stop_evt.is_set():
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(gpu_index)],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            if out:
                samples.append([x.strip() for x in out.split(",")])
        except Exception:
            pass
        stop_evt.wait(0.2)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
    sm = sorted(int(float(s[0])) for s in samples if s[0].replace(".", "").isdigit())
    mx = max(int(float(s[1])) for s in samples if s[1].replace(".", "").isdigit()) if samples else None
    reasons = set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in samples:
        for nm, val in zip(names, s[3:7]):
            if val.lower().startswith("active"):
                reasons.add(nm)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
            "samples": len(samples)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "library"],
                    help="ours | reference (unmodified upstream; unavailable offline) | library (reference-semantics "
                         "baseline: cuBLAS/SDPA through torch + per-tensor in-stream NCCL all-reduce, bench/torch_baseline.py)")
    ap.add_argument("--model", default="345M")
    ap.add_argument("--batch", type=int, default=4, help="sequences per GPU per step (reference config: 4)")
    ap.add_argument("--strategy", default="auto")
    ap.add_argument("--comm", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-exposed", action="store_true", help="skip the exposed-communication measurement (N > 1)")
    ap.add_argument("--no-tp", action="store_true", help="skip the tensor-parallel arm (N > 1)")
    ap.add_argument("--no-library-arm", action="store_true",
                    help="skip the same-box library comparator (cuBLAS / SDPA / per-tensor NCCL step, bench/torch_baseline.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (its loss, rank 0) as DIR/loss.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable":
                          "alibaba/TePDist is a Bazel-2.0 fork of mid-2020 TensorFlow (no setup.py/pyproject; CUDA 10/11, sm<=80); "
                          "pip install --no-index of /root/reference fails: not installable offline"}))
        return 0

    if os.environ.get("TEPDIST_HANG_DUMP"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["TEPDIST_HANG_DUMP"]), exit=True)
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from tepdist_b200 import ops
    from tepdist_b200.api import Trainer
    from tepdist_b200.models.gpt2 import CONFIGS, build_gpt2_graph

    W = max(args.warmup, 3)
    K = args.steps
    cfg = CONFIGS[args.model]
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    library = args.impl == "library"
    if library:
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "torch_baseline", os.path.join(os.path.dirname(os.path.abspath(__file__)), "bench", "torch_baseline.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        LibraryTrainer = mod.LibraryTrainer
        rank, world = int(os.environ.get("RANK", "0")), world_env
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
        torch.cuda.set_device(dev)
        if world > 1:
            dist.init_process_group("nccl", device_id=dev)
        lt = LibraryTrainer(cfg, dev, world, use_graph=not args.no_graph)
        step_dev = lambda tok, lab: lt.step(tok, lab)

        def step_host(tok, lab):
            return float(lt.step(tok.to(dev, non_blocking=True), lab.to(dev, non_blocking=True)))
        parallelism, local_rank = f"dp{world}", dev.index
    else:
        # weak scaling: the planner sees the GLOBAL step (batch = per-GPU batch x GPUs) and shards it; every rank then
        # feeds its own [per-GPU batch, seq] shard
        graph = build_gpt2_graph(cfg, batch=args.batch * world_env)
        trainer = Trainer(graph, strategy=args.strategy, use_cuda_graph=not args.no_graph, comm_mode=args.comm)
        rank, world = trainer.rank, trainer.world
        dev = trainer.device
        step_dev = lambda tok, lab: trainer.step_async({"tokens": tok, "labels": lab})
        step_host = lambda tok, lab: trainer.step({"tokens": tok, "labels": lab})
        local_rank = trainer.ctx["local_rank"]
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    B, S = args.batch, cfg.n_ctx
    is_pp = (not library) and args.strategy.startswith("pp")
    if is_pp:
        # pipeline plans: stage 0 consumes the tokens, the last stage the labels, each sliced per micro-batch -- every rank is
        # fed the GLOBAL batch (the same on all ranks) and the stage workers take what their stage needs
        args.no_exposed = args.no_tp = True
    gen = torch.Generator().manual_seed(1234 + (0 if is_pp else rank))
    # synthetic fake_input: random tokens, labels = tokens shifted by one (reference: examples/GPT2/inputs.py:42-55)
    nbuf = 4
    rows = B * world if is_pp else B
    host_tok = [torch.randint(0, cfg.n_vocab, (rows, S), generator=gen, dtype=torch.int32).pin_memory() for _ in range(nbuf)]
    host_lab = [torch.roll(t, -1, 1).pin_memory() for t in host_tok]
    dev_tok = [t.to(dev) for t in host_tok]
    dev_lab = [t.to(dev) for t in host_lab]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-timed region (inputs resident on device) ----------------
    for i in range(W):
        step_dev(dev_tok[i % nbuf], dev_lab[i % nbuf])
    barrier()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local_rank), daemon=True)
    if rank == 0:
        th.start()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    loss = None
    for i in range(K):
        loss = step_dev(dev_tok[i % nbuf], dev_lab[i % nbuf])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_count()
    final_loss = float(loss)
    if args.dump_outputs and rank == 0:
        # The step returns the loss and nothing else.  The weights it updates are not dumped: the gradient reductions add
        # with float atomics, and AdamW turns gradients at noise level (the attention key bias's is exactly zero) into
        # full-size updates, so the weights differ from run to run by far more than the loss does.
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "loss.npy"), loss.detach().float().reshape(-1).cpu().numpy())

    # ---------------- end-to-end through the public API: H2D inputs from pinned memory + D2H loss every step
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(K):
        step_host(host_tok[i % nbuf], host_lab[i % nbuf])
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    stop.set()

    # ---------------- exposed communication: the same sharded step with every collective replaced by a local stand-in
    # (TEPDIST_DRY_COMM, timing only); exposed comm = ms/step - ms/step(dry).  BASELINE.md north-star metric.
    ms_dry = 0.0
    if world > 1 and not library and not args.no_exposed:
        os.environ["TEPDIST_DRY_COMM"] = "1"
        dry = Trainer(graph, strategy=args.strategy, use_cuda_graph=not args.no_graph, comm_mode=args.comm)
        del os.environ["TEPDIST_DRY_COMM"]
        for i in range(W):
            dry.step_async({"tokens": dev_tok[i % nbuf], "labels": dev_lab[i % nbuf]})
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(K):
            dry.step_async({"tokens": dev_tok[i % nbuf], "labels": dev_lab[i % nbuf]})
        g1.record()
        barrier()
        ms_dry = g0.elapsed_time(g1)

    # ---------------- tensor-parallel arm (BASELINE.json config "GPT-2 345M auto-SPMD (tensor-parallel)"): the SAME global
    # step (batch = per-GPU batch x N) under the planner's Megatron plan (weight matrices stored sharded over all N GPUs,
    # `linear -> all_reduce -> + bias -> + residual` chains), once with the chains executed as GEMM -> NVLS all-reduce
    # (multimem kernels over the multicast-bound symmetric buffers, comm = fused) and once with NCCL collectives.
    tp_ms = {"fused": 0.0, "nccl": 0.0}
    tp_info = {}
    if world > 1 and not library and not args.no_tp:
        from tepdist_b200.runtime import executor as ex_mod
        for tag, fused, comm in (("fused", True, "fused"), ("nccl", False, "nccl")):
            try:
                ex_mod.TP_FUSED = fused
                ttr = Trainer(graph, strategy="tp", use_cuda_graph=not args.no_graph, comm_mode=comm)
                for i in range(W):
                    ttr.step_async({"tokens": dev_tok[i % nbuf], "labels": dev_lab[i % nbuf]})
                barrier()
                h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                h0.record()
                for i in range(K):
                    tl = ttr.step_async({"tokens": dev_tok[i % nbuf], "labels": dev_lab[i % nbuf]})
                h1.record()
                barrier()
                tp_ms[tag] = h0.elapsed_time(h1)
                tp_info[tag + "_chains"] = len(getattr(ttr.exec, "tp_fuse", {}) or {})
                tp_info[tag + "_loss"] = float(tl)
                tp_info["parallelism"] = ttr.plan_info.get("parallelism")
                del ttr
            except Exception as e:  # noqa: BLE001  (the headline number must survive a failure of the extra arm)
                tp_info[tag + "_error"] = f"{type(e).__name__}: {e}"[:300]
            finally:
                ex_mod.TP_FUSED = False

    # ---------------- pipeline: measured bubble per stage (2 extra steps with CUDA events around every stage body)
    pp_meas = None
    if is_pp:
        w = trainer.exec.worker
        w.timing = True
        bub = []
        for i in range(2):
            trainer.step_async({"tokens": dev_tok[i % nbuf], "labels": dev_lab[i % nbuf]})
            bub.append(w.last_timing["bubble"])
        w.timing = False
        tb = torch.tensor([sum(bub) / len(bub), float(w.stage)], dtype=torch.float64, device=dev)
        allb = [torch.zeros_like(tb) for _ in range(world)]
        dist.all_gather(allb, tb)
        per_stage = {}
        for x in allb:
            per_stage.setdefault(int(x[1].item()), []).append(float(x[0].item()))
        pp_meas = {"bubble_per_stage": {str(k): round(sum(v) / len(v), 4) for k, v in sorted(per_stage.items())},
                   "cuda_graph": bool(w.use_graph), "graphs_captured": w.graph_stats["captured"], "slots": w.num_slots}

    # ---------------- same-box comparator: the library step (cuBLAS GEMMs, SDPA attention, torch fused AdamW, one in-stream
    # ncclAllReduce per gradient tensor, whole step in a CUDA graph; none of this repository's kernels) timed in THIS process on
    # THIS box, so the ratio does not depend on box-to-box variance (the reference itself cannot be installed: DESIGN.md)
    ms_lib = 0.0
    lib_err = None
    if not library and not is_pp and not args.no_library_arm and cfg.name == "gpt2-345M":
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location(
                "torch_baseline", os.path.join(os.path.dirname(os.path.abspath(__file__)), "bench", "torch_baseline.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            lt = mod.LibraryTrainer(cfg, dev, world, use_graph=not args.no_graph)
            for i in range(W):
                lt.step(dev_tok[i % nbuf], dev_lab[i % nbuf])
            barrier()
            l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0.record()
            for i in range(K):
                lt.step(dev_tok[i % nbuf], dev_lab[i % nbuf])
            l1.record()
            barrier()
            ms_lib = l0.elapsed_time(l1)
            del lt
        except Exception as e:  # noqa: BLE001
            lib_err = f"{type(e).__name__}: {e}"[:300]

    t = torch.tensor([ms, ms_e2e, ms_dry, tp_ms["fused"], tp_ms["nccl"], ms_lib], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_dry, tp_fused_ms, tp_nccl_ms, ms_lib = t.tolist()
    if rank == 0:
        tokens = B * S * world * K
        value = tokens / (ms / 1e3)
        e2e = tokens / (ms_e2e / 1e3)
        fl = cfg.flops_per_token() * value
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")))
        except Exception:
            pass
        out = {
            "metric": "GPT-2 tokens/sec (whole job, device-timed, max over ranks)", "value": value, "unit": "tokens/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (value / REF_BASELINE_TOKENS_PER_S) if REF_BASELINE_TOKENS_PER_S else None,
            "dtype": "bf16", "data": "synthetic (random tokens, labels=shift; random-init weights)",
            "impl": "library-baseline (torch cuBLAS/SDPA kernels, per-tensor NCCL all-reduce in-stream, no kernels of this repo)" if library else "ours",
            "config": {"model": cfg.name, "n_layer": cfg.n_layer, "n_embd": cfg.n_embd, "n_head": cfg.n_head,
                       "global_batch": B * world, "per_gpu_batch": B, "seq_len": S, "vocab": cfg.n_vocab,
                       "optimizer": "AdamW (fp32 master + moments)", "parallelism": parallelism if library else trainer.plan_info.get("parallelism", f"dp{world}"),
                       "cuda_graph": (lt.use_graph if library else not args.no_graph), "comm": "nccl-per-tensor" if library else args.comm,
                       "l2": "working set per step >> 126 MB L2 (0.7 GB bf16 weights + 5.7 GB fp32 optimizer state touched every step)"},
            "e2e": {"value": e2e, "unit": "tokens/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": 2 * rows * S * 4 * world, "d2h_bytes_per_step": 4 * world},
            "gpu_launches": launches,
            "exposed_comm_ms_per_step": ((ms - ms_dry) / K) if ms_dry > 0 else (0.0 if world == 1 else None),
            "compute_only_ms_per_step": (ms_dry / K) if ms_dry > 0 else None,
            "model_tflops_per_gpu": fl / world / 1e12,
            "mfu_of_measured_sustained_peak": (fl / world / 1e12) / peaks["bf16_tflops_sustained"] if peaks.get("bf16_tflops_sustained") else None,
            "final_loss": final_loss,
            "clocks": summarize_clocks(samples),
        }
        if args.dump_outputs:
            out["dump_outputs"] = {"dir": args.dump_outputs, "arrays": ["loss"]}
        if ms_lib > 0:
            out["library_arm"] = {"ms_per_step": ms_lib / K, "tokens_per_s": tokens / (ms_lib / 1e3), "ours_over_library": ms_lib / ms,
                                  "what": "same box, same process: torch cuBLAS / SDPA / fused AdamW + per-tensor in-stream NCCL all-reduce, CUDA graph"}
        elif lib_err:
            out["library_arm"] = {"error": lib_err}
        if is_pp:
            pi = trainer.plan_info
            out["pipeline"] = {"stages": pi.get("stages"), "micro_batches": pi.get("micro"), "spmd": pi.get("spmd"),
                               "stage_cut": pi.get("stage_method"), "cut_bytes": pi.get("cut_bytes"),
                               "scheduler_bubble_estimate": pi.get("bubble_est"), "scheduler_makespan_estimate_s": pi.get("makespan_est"),
                               "p2p": "NCCL isend/irecv on side streams", **(pp_meas or {})}
            out["pipeline"]["measured_bubble_mean"] = (sum(out["pipeline"]["bubble_per_stage"].values()) /
                                                        max(1, len(out["pipeline"]["bubble_per_stage"]))) if pp_meas else None
        if world > 1 and not library and not args.no_tp:
            tp = dict(tp_info)
            tp["global_batch"] = B * world
            for tag, v in (("fused", tp_fused_ms), ("nccl", tp_nccl_ms)):
                if v > 0:
                    tp[tag + "_ms_per_step"] = v / K
                    tp[tag + "_tokens_per_s"] = tokens / (v / 1e3)
            if tp_fused_ms > 0 and tp_nccl_ms > 0:
                tp["fused_over_nccl"] = tp_nccl_ms / tp_fused_ms
            tp["note"] = ("same global batch as the data-parallel headline; fused = GEMM -> multimem (NVLS) all-reduce with bias + "
                          "residual in the reduction kernel, nccl = same plan with NCCL all-reduce + separate bias / residual adds")
            out["tp"] = tp
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        # NCCL communicators captured inside CUDA graphs do not tear down cleanly (destroy_process_group blocks):
        # everything is flushed, leave without running destructors
        sys.stdout.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
