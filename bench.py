#!/usr/bin/env python
"""Headline benchmark: DLRM (Criteo-1TB shape, 26 sparse + 13 dense, MLPerf arch) training
throughput in samples/s, whole job, device timed, max over ranks.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 20 --warmup 5
    python bench.py --impl reference ...        # unmodified reference from baseline/_ref (if installable)

Prints ONE JSON line on rank 0 (see README / DESIGN.md for the field contract).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from typing import Any, Dict, List, Optional

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Criteo-1TB categorical cardinalities with the MLPerf 40M row cap (26 features)
CRITEO_1TB_40M = [39884406, 39043, 17289, 7420, 20263, 3, 7120, 1543, 63, 38532951, 2953546, 403346, 10, 2208, 11938, 155, 4, 976, 14,
                  39979771, 25641295, 39664984, 585935, 12972, 108, 36]
HOST_HEAD_STEPS = 16  # host enqueue time is averaged over this many steps right after the start barrier
BASELINE_SAMPLES_PER_SEC = {1: 50_000.0, 8: 350_000.0}  # reference published numbers (A100), BASELINE.md
DUMP_BYTES = 64 << 20  # --dump-outputs budget over all ranks


def parse_args() -> argparse.Namespace:
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    p.add_argument("--batch-size", type=int, default=int(os.environ.get("TRB_BENCH_BATCH", 32768)), help="per-GPU batch (weak scaling)")
    p.add_argument("--embedding-dim", type=int, default=128)
    p.add_argument("--dense-arch", type=str, default="512,256,128")
    p.add_argument("--over-arch", type=str, default="1024,1024,512,256,1")
    p.add_argument("--row-cap", type=int, default=int(os.environ.get("TRB_BENCH_ROW_CAP", 40_000_000)))
    p.add_argument("--pooling", type=int, default=1, help="ids per sparse feature (Criteo is one-hot)")
    p.add_argument("--lr", type=float, default=0.01)
    p.add_argument("--config", type=str, default="dlrm", choices=["dlrm", "rw100m", "dcn_cw", "two_tower"],
                   help="BASELINE.json configs: dlrm = #2 (table-wise DLRM, the headline); rw100m = #3 (one 100 M-row table row-wise); "
                        "dcn_cw = #4 (DLRM-DCNv2, column-wise tables, + fp8 quantized inference QPS); two_tower = #5 (retrieval, planner-driven table-row-wise)")
    p.add_argument("--sharding", type=str, default="auto", choices=["auto", "planner", "table_wise", "row_wise", "column_wise"],
                   help="auto / planner: EmbeddingShardingPlanner under the config's sharding-type constraint (the SAME rule the reference arm "
                        "uses: table_wise for the headline); table_wise / row_wise / column_wise: hand-made plans")
    p.add_argument("--overlap-sparse", type=int, default=int(os.environ.get("TRB_BENCH_OVERLAP", 1)),
                   help="1: embedding arch on a side stream (forward beside the bottom MLP, gradient push + fused optimizer beside the bottom MLP backward)")
    p.add_argument("--measure-comm", type=int, default=1, help="N > 1: time the NVLink phases in isolation after the run (exposed all-to-all ms, GB/s)")
    p.add_argument("--dense-backend", type=str, default=os.environ.get("TRB_DENSE_BACKEND", "auto"))
    p.add_argument("--transport", type=str, default=os.environ.get("TRB_TRANSPORT", "auto"), help="auto | p2p | nccl")
    p.add_argument("--dp-rows", type=int, default=int(os.environ.get("TRB_BENCH_DP_ROWS", 0)),
                   help="--sharding table_wise only: tables with at most this many rows are data-parallel when N > 1 (0 = every table model-parallel)")
    p.add_argument("--cuda-graphs", type=int, default=int(os.environ.get("TRB_BENCH_GRAPHS", -1)),
                   help="1 (= -1, the default): replay the dense sub-modules as CUDA graphs (host enqueue 1.6-2.6 ms -> 0.74 ms per step; "
                        "end to end 15.4 M -> 17.7 M samples/s on one GPU); 0: eager")
    p.add_argument("--profile-host", action="store_true", help="cProfile 10 extra steps on rank 0 (stderr)")
    p.add_argument("--ddp-bucket-mb", type=float, default=float(os.environ.get("TRB_BENCH_DDP_BUCKET_MB", 2)), help="DDP gradient bucket size of the dense part")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--phase-times", action="store_true", help="diagnostics: forward / backward / optimizer device time of the plain step (stderr)")
    p.add_argument("--trace-e2e", type=str, default="", help="diagnostics: torch.profiler trace (chrome json + op table) of 6 extra pipeline steps")
    p.add_argument("--num-host-batches", type=int, default=8)
    p.add_argument("--dump-outputs", type=str, default="", metavar="DIR",
                   help="write what the last timed step returned (loss, logits, labels) as DIR/<name>.npy in float32, to compare two builds "
                        "output for output; with several GPUs each rank writes <name>_rank<r>.npy")
    return p.parse_args()


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int) -> None:
        self.gpu = gpu_index
        self.proc: Optional[subprocess.Popen] = None
        self.lines: List[str] = []
        self._t: Optional[threading.Thread] = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def reader() -> None:
            assert self.proc is not None and self.proc.stdout is not None
            for line in self.proc.stdout:
                self.lines.append((time.time(), line.strip()))

        self._t = threading.Thread(target=reader, daemon=True)
        self._t.start()

    def mark_start(self) -> None:
        """The sampler is started before warm-up (nvidia-smi takes longer to start than a short timed region lasts);
        only samples that arrive between mark_start() and stop() are reported."""
        self.t0 = time.time()

    def stop(self) -> Dict[str, Any]:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = getattr(self, "t0", 0.0)
        inside = [ln for ts, ln in self.lines if t0 <= ts <= t1 + 0.11]
        window = "timed"
        if not inside:  # region shorter than one sampling period: fall back to the closest samples taken under (warm-up) load
            inside = [ln for ts, ln in self.lines][-3:]
            window = "warmup+timed"
        self.window = window
        for ln in inside:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "window": getattr(self, "window", "timed")}


def reference_arm(args: argparse.Namespace) -> None:
    """Run the UNMODIFIED reference from baseline/_ref if it is importable; otherwise say why."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    why = None
    if not os.path.isdir(ref):
        why = "baseline/_ref missing (reference not installed: fbgemm_gpu wheel unavailable offline, see DESIGN.md)"
    else:
        sys.path.insert(0, ref)
        try:
            import torchrec  # noqa: F401
        except Exception as e:  # fbgemm_gpu hard import
            why = f"reference import failed: {type(e).__name__}: {str(e).splitlines()[0][:160]}"
    if why is not None:
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": why}))
        return
    from baseline.run_reference import run as run_reference  # type: ignore

    run_reference(args)


def build_ours(args: argparse.Namespace, device, rank: int, world: int):
    """Model + plan + optimizer of the selected BASELINE config. Returns (dmp, opt, keys, hashes, ids_per_feature, num_dense, backend, info)."""
    import torch
    import torch.distributed as dist

    from torchrec_b200.models.dlrm import DLRM, DLRM_DCN, DLRMTrain
    from torchrec_b200.modules.embedding_configs import EmbeddingBagConfig
    from torchrec_b200.modules.embedding_modules import EmbeddingBagCollection
    from torchrec_b200.ops import dense as _dense
    from torchrec_b200.optim.apply_optimizer_in_backward import apply_optimizer_in_backward
    from torchrec_b200.optim.keyed import CombinedOptimizer, KeyedOptimizerWrapper
    from torchrec_b200.optim.optimizers import in_backward_optimizer_filter
    from torchrec_b200.optim.rowwise_adagrad import RowWiseAdagrad
    from torchrec_b200.parallel import sharding_plan as sp
    from torchrec_b200.parallel.embeddingbag import EmbeddingBagCollectionSharder
    from torchrec_b200.parallel.model_parallel import DistributedModelParallel
    from torchrec_b200.parallel.planner import EmbeddingShardingPlanner, Topology
    from torchrec_b200.parallel.planner.types import ParameterConstraints
    from torchrec_b200.parallel.types import ShardingPlan

    cfg = args.config
    D = args.embedding_dim
    num_dense = 13
    if cfg == "two_tower":
        keys, hashes, num_dense = ["user", "item"], [min(40_000_000, args.row_cap), min(10_000_000, args.row_cap)], 1
    else:
        hashes = [min(h, args.row_cap) for h in CRITEO_1TB_40M]
        keys = [f"cat_{i}" for i in range(26)]
        if cfg == "rw100m":
            hashes[0] = 100_000_000
    tables = [EmbeddingBagConfig(name=f"t_{k}", embedding_dim=D, num_embeddings=h, feature_names=[k]) for k, h in zip(keys, hashes)]
    ebc = EmbeddingBagCollection(tables=tables, device=torch.device("meta"))
    apply_optimizer_in_backward(RowWiseAdagrad, ebc.parameters(), {"lr": args.lr, "eps": 1e-8})
    dense_arch = [int(x) for x in args.dense_arch.split(",")]
    over_arch = [int(x) for x in args.over_arch.split(",")]
    if cfg == "two_tower":
        from examples.two_tower_retrieval import TwoTower, TwoTowerTrainTask

        model = TwoTowerTrainTask(TwoTower(ebc, [256, 128], device=device))
        module_path = "two_tower.ebc"
    elif cfg == "dcn_cw":
        model = DLRMTrain(DLRM_DCN(ebc, 13, dense_arch, over_arch, dcn_num_layers=3, dcn_low_rank_dim=512, dense_device=device))
        module_path = "model.sparse_arch.embedding_bag_collection"
    else:
        model = DLRMTrain(DLRM(ebc, 13, dense_arch, over_arch, dense_device=device))
        module_path = "model.sparse_arch.embedding_bag_collection"

    backend = args.dense_backend
    if backend == "auto":
        backend = os.environ.get("TRB_DENSE_DEFAULT", "tcgen05")  # bf16 tensor-core dense path is the product
    _dense.set_dense_backend(backend)
    # bf16 pooled embeddings (half the NVLink / HBM bytes) when the dense arch computes in bf16
    fused_params = {"output_dtype": torch.bfloat16} if backend == "tcgen05" else None
    sharder = EmbeddingBagCollectionSharder(fused_params=fused_params)

    # sharding-type constraint of the config (identical rule in the reference arm: baseline/run_reference.py)
    rule = {"dlrm": "table_wise", "rw100m": "table_wise", "dcn_cw": "column_wise", "two_tower": "table_row_wise"}[cfg]
    per_table = {t.name: rule for t in tables}
    if cfg == "rw100m":
        per_table[tables[0].name] = "row_wise"
    if world == 1:  # one rank: every sharding type degenerates to the whole table on rank 0
        per_table = {t.name: "table_wise" for t in tables}
    mode = args.sharding if args.sharding != "auto" else "planner"
    info = {"plan": mode, "rule": rule if cfg != "rw100m" else "row_wise(t_cat_0: 100 M rows) + table_wise"}
    if mode == "planner":
        cw_shards = min(world, 4)
        constraints = {t.name: ParameterConstraints(sharding_types=[per_table[t.name]], compute_kernels=["fused"],
                                                    **({"min_partition": max(32, D // cw_shards)} if per_table[t.name] == "column_wise" else {})) for t in tables}
        # table-row-wise needs "hosts": on one 8-GPU NVSwitch box the two halves play the hosts (a table lives on one half, row-wise inside it)
        local_world = world if rule != "table_row_wise" or world < 4 else world // 2
        info["topology"] = f"{world} ranks, local_world_size {local_world}"
        planner = EmbeddingShardingPlanner(topology=Topology(world_size=world, local_world_size=local_world, compute_device="cuda"), batch_size=args.batch_size,
                                           constraints=constraints)
        if world > 1:
            plan = planner.collective_plan(model, [sharder], dist.GroupMember.WORLD)
        else:
            plan = planner.plan(model, [sharder])
        placed = plan.plan[module_path]
        info["tables_per_rank"] = [sum(1 for ps in placed.values() if r in (ps.ranks or [])) for r in range(world)]
    else:
        if mode == "table_wise":
            # greedy balance: bytes first (big tables spread), then lookups per rank
            load = [[0.0, 0] for _ in range(world)]
            gens = {}
            order = sorted(range(len(tables)), key=lambda i: -hashes[i])
            tot = float(sum(hashes))
            if world > 1 and args.dp_rows > 0:
                tiny = [i for i in order if hashes[i] <= args.dp_rows]
                for i in tiny:
                    gens[tables[i].name] = sp.data_parallel()
                order = [i for i in order if i not in tiny]
            for i in order:
                r = min(range(world), key=lambda r: (load[r][0] / tot * world + load[r][1] / len(tables) * world, r))
                load[r][0] += hashes[i]
                load[r][1] += 1
                gens[tables[i].name] = sp.table_wise(rank=r)
        elif mode == "row_wise":
            gens = {t.name: sp.row_wise() for t in tables}
        else:
            gens = {t.name: (sp.column_wise(ranks=[(i + j) % world for j in range(min(world, 4))]) if world > 1 else sp.table_wise(rank=0)) for i, t in enumerate(tables)}
        mplan = sp.construct_module_sharding_plan(ebc, gens, sharder=sharder, world_size=world, local_size=world, device_type="cuda")
        plan = ShardingPlan({module_path: mplan})
    # data-parallel wrapping is deferred (main() calls dmp.init_data_parallel()) so that CUDA graphs of the dense sub-modules can
    # be captured first: DDP keeps the parameters' AccumulateGrad nodes alive on the default stream, which a capture may not touch
    # small DDP buckets: the dense gradients of the top MLP are reduced while the embedding backward + bottom MLP backward still run; with the
    # default 25 MB cap everything but the last layer waits in ONE bucket for the very last gradient and the all-reduce (239 us at 8 GPUs in
    # profiles/step_kernels_n8_r2.md) sits exposed at the end of the step
    from torchrec_b200.parallel.model_parallel import DefaultDataParallelWrapper

    dmp = DistributedModelParallel(model, device=device, plan=plan, sharders=[sharder], init_data_parallel=False,
                                   data_parallel_wrapper=DefaultDataParallelWrapper(bucket_cap_mb=args.ddp_bucket_mb))
    dense_opt = KeyedOptimizerWrapper(dict(in_backward_optimizer_filter(dmp.named_parameters())), lambda params: torch.optim.SGD(params, lr=args.lr))
    opt = CombinedOptimizer([dmp.fused_optimizer, dense_opt])
    return dmp, opt, keys, hashes, [args.pooling] * len(keys), num_dense, backend, info


def find_planes(module) -> list:
    """NVLink sparse planes created by the sharded modules of ``module`` (one per batch size / id source)."""
    out = []
    for m in module.modules():
        eng = getattr(m, "_engine", None)
        if eng is not None:
            out.extend(eng.__dict__.get("_planes", {}).values())
    return out


def measure_comm(dmp, device, world: int, iters: int = 10) -> Optional[Dict[str, Any]]:
    """Times the NVLink phases of the sparse plane in isolation (CUDA events, every rank in lock step, max over ranks) on the ids of
    the last batch: the fused lookup + output dist against the SAME lookup writing locally (difference = exposed forward all-to-all),
    the gradient push (pure communication) and the input dist. Bytes are what this rank stores into peer memory per step."""
    import torch
    import torch.distributed as dist

    planes = [p for p in find_planes(dmp) if p.capacity > 0 and p.W > 1]
    if not planes:
        return None
    pl = planes[0]
    slot = (pl.step - 1) % pl.N_ID_SLOTS
    reg = pl.regions(slot)
    esz = torch.empty(0, dtype=pl.wire_dtype).element_size()
    my_cols = sum(u.shard.cols for u in pl.eng._local_units)
    sent_fwd = (world - 1) * pl.B_local * my_cols * esz                 # pooled rows of MY units for the other ranks' samples
    sent_bwd = pl.B_local * (pl.total_cols - my_cols) * esz             # gradient columns of the OTHER ranks' units
    grad = torch.randn(pl.B_local, pl.total_cols, device=device).to(pl.wire_dtype)

    def timed(fn) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fn()
        dist.barrier()
        torch.cuda.synchronize()
        pl.group.barrier(0)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def fwd_fused():
        pl._forward_kernels(reg, 1)
        pl.group.barrier(0)

    def fwd_local():
        pl._forward_kernels(reg, 1, local_only=True)
        pl.group.barrier(0)

    def push():
        pl._push_kernels(grad)
        pl.group.barrier(0)

    t_fused, t_local, t_push = timed(fwd_fused), timed(fwd_local), timed(push)
    t_barrier = timed(lambda: pl.group.barrier(0))
    res = {"fwd_fused_lookup_dist_ms": t_fused, "fwd_same_lookup_local_ms": t_local, "bwd_grad_push_ms": t_push, "device_barrier_ms": t_barrier,
           "fwd_sent_bytes_per_rank": sent_fwd, "bwd_sent_bytes_per_rank": sent_bwd,
           "fwd_gbps": sent_fwd / (t_fused * 1e-3) / 1e9, "bwd_gbps": sent_bwd / (max(t_push - t_barrier, 1e-6) * 1e-3) / 1e9,
           "exposed_fwd_ms": max(0.0, t_fused - t_local), "exposed_bwd_ms": t_push, "nvlink_peak_gbps": 900.0, "nvlink_measured_peer_copy_gbps": 770.0}
    return res


def fp8_inference_qps(args, dmp, device, rank: int, world: int, keys, hashes) -> Dict[str, Any]:
    """Config #4 tail: quantize the tables to block-scaled FP8 (e4m3 + one fp16 scale per 32 elements) and time the serving
    lookup (quantized table-batched kernel, bf16 output) on this GPU: fresh tables of the same shapes (the trained shards live on
    other ranks), one-hot ids, device-timed."""
    import torch

    from torchrec_b200.ops.quant_tbe import QuantTableBatchedEmbeddingBags
    from torchrec_b200.types import DataType

    rows = [min(h, 4_000_000) for h in hashes]
    B = args.batch_size
    q = QuantTableBatchedEmbeddingBags([(f"t{i}", r, args.embedding_dim, DataType.FP8) for i, r in enumerate(rows)], output_dtype=torch.bfloat16, device=device)
    q.weights.random_(0, 120)  # arbitrary finite e4m3 payloads / scales: the timing does not depend on the values
    g = torch.Generator(device="cpu").manual_seed(7)
    # 16 distinct batches: 16 x 26 x 32768 rows x 144 B = 1.9 GB of gathered rows, far beyond the 126 MB L2 (no batch is re-read from cache)
    id_sets = [torch.cat([torch.randint(0, r, (B,), generator=g) for r in rows]).to(device) for _ in range(16)]
    off = torch.arange(0, len(rows) * B + 1, device=device, dtype=torch.int64)
    for i in range(4):
        q(id_sets[i], off)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    n = 32
    for i in range(n):
        out = q(id_sets[i % len(id_sets)], off)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    row_bytes = args.embedding_dim + args.embedding_dim // 32 * 2
    return {"format": "FP8_BLOCK (e4m3, fp16 scale / 32 elems)", "samples_per_s_per_gpu": B / (ms * 1e-3), "ms_per_batch": ms,
            "table_bytes": int(sum(rows)) * row_bytes, "gathered_gbps": len(rows) * B * row_bytes / (ms * 1e-3) / 1e9,
            "hbm_gbps_rows_plus_bf16_output": len(rows) * B * (row_bytes + args.embedding_dim * 2) / (ms * 1e-3) / 1e9,
            "l2_policy": "16 distinct one-hot batches (1.9 GB of rows) cycled: no batch is served from the 126 MB L2", "out_shape": list(out.shape)}


def dump_outputs(directory: str, arrays: Dict[str, Any], rank: int, world: int) -> None:
    """Writes one step's outputs as float32 ``<name>.npy`` files. All ranks together write at most DUMP_BYTES: when the per-sample
    arrays are longer than this rank's share, the same fixed, seeded sample of samples is kept from every array."""
    import numpy as np
    import torch

    host = {k: v.detach().float().reshape(-1).cpu() for k, v in arrays.items()}
    n = max(t.numel() for t in host.values())
    cap = DUMP_BYTES // (4 * len(host) * world)
    if n > cap:
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values
        host = {k: t[keep] if t.numel() == n else t for k, t in host.items()}
    os.makedirs(directory, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    for k, t in host.items():
        np.save(os.path.join(directory, f"{k}{suffix}.npy"), t.numpy())


def main() -> None:
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    from torchrec_b200.datasets.random import RandomRecDataset
    from torchrec_b200.ops import _lib
    from torchrec_b200.parallel.train_pipeline import TrainPipelineSparseDist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    device = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(device)
    if os.environ.get("TRB_BENCH_BIND_NUMA", "1") != "0":
        from torchrec_b200.utils.affinity import bind_to_gpu_numa

        _bound = bind_to_gpu_numa(local_rank)  # pinned staging buffers + launch threads on the GPU's socket (H2D does not cross sockets)
        globals()["_CPU_BINDING"] = f"{len(_bound)} NUMA-local cpus" if _bound else "unchanged"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        pg_opts = None
        try:  # collectives of the dense gradients must not queue behind the long embedding kernels
            pg_opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            pass
        dist.init_process_group(backend="nccl", device_id=device, pg_options=pg_opts)
    if args.transport != "auto":
        os.environ["TRB_TRANSPORT"] = args.transport  # "nccl": the internal UNFUSED arm (own lookup kernels + NCCL all-to-alls)
    _lib.lib()

    torch.manual_seed(0)  # model initialisation, like the batches below, is the same in every run with the same arguments
    dmp, opt, keys, hashes, ids_per_feature, num_dense, dense_backend, plan_info = build_ours(args, device, rank, world)
    B = args.batch_size
    ds = RandomRecDataset(keys, B, hash_sizes=hashes, ids_per_features=ids_per_feature, num_dense=num_dense, manual_seed=1234 + rank,
                          num_generated_batches=args.num_host_batches, pin_memory=True)
    host_batches = ds.batch_generator._generated_batches
    dev_batches = [b.to(device) for b in host_batches]
    torch.cuda.synchronize()

    if args.cuda_graphs < 0:
        args.cuda_graphs = 1
    if not args.cuda_graphs:
        dmp.init_data_parallel()
    inner = getattr(dmp.module, "model", None)
    if args.cuda_graphs and hasattr(inner, "capture_dense_graphs"):
        # the dense sub-modules (bottom MLP, interaction + top MLP + head) replay as CUDA graphs: their ~50 launches and ~100 ATen
        # calls per step made the step launch-bound once DDP / NVLink dists were added (host enqueue 2.0 ms vs 2.1 ms of GPU time)
        with torch.no_grad():
            sample_emb = inner.sparse_arch(dev_batches[0].sparse_features)
        inner.capture_dense_graphs(dev_batches[0].dense_features, sample_emb)
        inner.overlap_sparse_dense = bool(args.overlap_sparse)
        torch.cuda.synchronize()
        dmp.init_data_parallel()
    elif args.cuda_graphs:
        args.cuda_graphs = 0
        dmp.init_data_parallel()

    def step(batch):
        opt.zero_grad()
        loss, out = dmp(batch)
        loss.backward()
        opt.step()
        return loss, out

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (kernel-side number) ----------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        step(dev_batches[i % len(dev_batches)])
    barrier()
    sampler.mark_start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    t_host0 = time.perf_counter()
    t_host_head = None
    for i in range(args.steps):
        loss, out = step(dev_batches[i % len(dev_batches)])
        if i == HOST_HEAD_STEPS - 1:
            t_host_head = time.perf_counter()
    # CPU time to ENQUEUE a step (>= ms_per_step means launch-bound). Measured over the first steps after the barrier: once the host
    # runs ~1000 launches ahead the driver blocks it and the average over the whole run just converges to the device time
    host_ms = ((t_host_head or time.perf_counter()) - t_host0) * 1e3 / (HOST_HEAD_STEPS if t_host_head else args.steps)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - n0
    if args.dump_outputs:  # before any further step: with CUDA graphs the logits live in a buffer the next replay overwrites
        dump_outputs(args.dump_outputs, {"loss": loss, "logits": out[1], "labels": out[2]}, rank, world)
    if args.phase_times:  # diagnostics: where the device time of the plain step goes (events on the main stream, no profiler attached)
        n_ph = 20
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(n_ph)]
        for i in range(n_ph):
            b = dev_batches[i % len(dev_batches)]
            evs[i][0].record()
            opt.zero_grad()
            loss_p, _ = dmp(b)
            evs[i][1].record()
            loss_p.backward()
            evs[i][2].record()
            opt.step()
            evs[i][3].record()
        torch.cuda.synchronize()
        ph = [sum(evs[i][k].elapsed_time(evs[i][k + 1]) for i in range(4, n_ph)) / (n_ph - 4) for k in range(3)]
        gap = sum(evs[i][3].elapsed_time(evs[i + 1][0]) for i in range(4, n_ph - 1)) / (n_ph - 5)
        sys.stderr.write("phase_ms " + json.dumps({"forward": ph[0], "backward": ph[1], "optimizer": ph[2], "between_steps": gap, "rank": rank}) + "\n")
    clocks = sampler.stop()
    if world > 1:  # worst GPU of the job: lowest median SM clock, union of throttle reasons
        allc: List[Any] = [None] * world
        dist.all_gather_object(allc, clocks)
        ok = [c for c in allc if c.get("sm_mhz") is not None]
        if ok:
            clocks = dict(min(ok, key=lambda c: c["sm_mhz"]))
            clocks["reasons"] = sorted({r for c in allc for r in c.get("reasons", [])})
            clocks["samples"] = sum(c.get("samples", 0) for c in ok)
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = B * world * args.steps / (ms_max / 1e3)

    # ---------------- end-to-end through the public pipeline API ------------------------------------
    e2e: Optional[Dict[str, Any]] = None
    if not args.no_e2e:
        late = bool(int(os.environ.get("TRB_BENCH_LATE_DIST", "1")))
        pipe = TrainPipelineSparseDist(dmp, opt, device, data_dist_after_forward=late, enqueue_batch_after_forward=late)

        def host_iter(n: int):
            for i in range(n):
                yield host_batches[i % len(host_batches)]

        loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        total = max(args.warmup, 3) + args.steps
        it = host_iter(total + 2)
        for _ in range(max(args.warmup, 3)):
            out = pipe.progress(it)
        barrier()
        e0.record()
        t_e2e0 = time.perf_counter()
        t_e2e_head = None
        for i in range(args.steps):
            out = pipe.progress(it)
            loss_host.copy_(out[0].detach().reshape(1), non_blocking=True)  # D2H read of the step's loss
            if i == HOST_HEAD_STEPS - 1:
                t_e2e_head = time.perf_counter()
        e2e_host_ms = ((t_e2e_head or time.perf_counter()) - t_e2e0) * 1e3 / (HOST_HEAD_STEPS if t_e2e_head else args.steps)
        e1.record()
        barrier()
        ms2 = e0.elapsed_time(e1)
        t2 = torch.tensor([ms2], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e = {"value": B * world * args.steps / (float(t2.item()) / 1e3), "unit": "samples/s",
               "h2d_bytes_per_step": host_batches[0].nbytes(), "d2h_bytes_per_step": 4, "ms_per_step": float(t2.item()) / args.steps, "host_enqueue_ms_per_step": e2e_host_ms,
               "loss": float(loss_host.item())}

    if args.trace_e2e and not args.no_e2e:
        from torch.profiler import ProfilerActivity, profile

        it3 = host_iter(6 + 4)
        for _ in range(2):
            pipe.progress(it3)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(4):
                out = pipe.progress(it3)
                loss_host.copy_(out[0].detach().reshape(1), non_blocking=True)
            torch.cuda.synchronize()
        if rank == 0:
            # compact per-kernel timeline of the LAST profiled step (stream, start us, duration us, name): what overlaps what
            try:
                evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time_total > 0]
                evs.sort(key=lambda e: e.time_range.start)
                marks = [e.time_range.start for e in evs if "interaction_fwd" in e.name]
                t_from = marks[-1] - 400 if marks else (evs[0].time_range.start if evs else 0)
                with open(args.trace_e2e + ".timeline.txt", "w") as f:
                    for e in evs:
                        if e.time_range.start >= t_from:
                            f.write("%10.1f %8.1f  %s\n" % (e.time_range.start - t_from, e.time_range.elapsed_us(), e.name[:100]))
            except Exception as ex:  # diagnostics only
                sys.stderr.write(f"timeline dump failed: {ex}\n")
            prof.export_chrome_trace(args.trace_e2e)
            with open(args.trace_e2e + ".txt", "w") as f:
                f.write(prof.key_averages().table(sort_by="self_cpu_time_total", row_limit=45, max_name_column_width=70))
                f.write("\n\n")
                f.write(prof.key_averages().table(sort_by="self_cuda_time_total", row_limit=70, max_name_column_width=90))
    if args.profile_host:
        # where does the host time of a step go? (diagnostics only; every rank runs the same steps: the NVLink barriers are collective)
        import cProfile
        import io
        import pstats

        def profiled(label, fn, n=10):
            pr = cProfile.Profile() if rank == 0 else None
            if pr is not None:
                pr.enable()
            for i in range(n):
                fn(i)
            if pr is not None:
                pr.disable()
                torch.cuda.synchronize()
                for key in ("tottime", "cumulative"):
                    buf = io.StringIO()
                    pstats.Stats(pr, stream=buf).sort_stats(key).print_stats(40)
                    sys.stderr.write(f"==== host profile: {label} ({n} steps), sorted by {key}\n" + buf.getvalue())
            torch.cuda.synchronize()

        if rank == 0:
            torch.cuda.set_sync_debug_mode("warn")  # every host<->stream synchronisation inside a step is reported on stderr
        for i in range(2):
            step(dev_batches[i % len(dev_batches)])
        torch.cuda.set_sync_debug_mode("default")
        profiled("plain step", lambda i: step(dev_batches[i % len(dev_batches)]))
        if not args.no_e2e:
            it2 = host_iter(10 + 4)
            profiled("TrainPipelineSparseDist.progress", lambda i: pipe.progress(it2))
    comm = None
    if world > 1 and args.measure_comm and args.transport != "nccl":
        comm = measure_comm(dmp, device, world)
    extra: Dict[str, Any] = {}
    if args.config == "dcn_cw":
        extra["fp8_inference"] = fp8_inference_qps(args, dmp, device, rank, world, keys, hashes)
    planes = find_planes(dmp)
    if rank == 0:
        base = BASELINE_SAMPLES_PER_SEC.get(world) if args.config == "dlrm" else None
        out = {
            "metric": "DLRM training throughput (samples/s, whole job, device-timed, max over ranks)",
            "value": value,
            "unit": "samples/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": (value / base) if base else None,
            "dtype": "bf16" if dense_backend == "tcgen05" else "fp32",
            "data": "synthetic (random Criteo-1TB-shaped ids/dense, random-init tables)",
            "impl": "ours",
            "config": {
                "name": args.config,
                "model": {"dlrm": "DLRM", "rw100m": "DLRM", "dcn_cw": "DLRM-DCNv2 (3 cross layers, rank 512)", "two_tower": "two-tower retrieval (examples/two_tower_retrieval.py)"}[args.config]
                         + " (%d sparse x dim %d, dense %s, over %s), fp32 tables + fused row-wise Adagrad, dense SGD" % (len(keys), args.embedding_dim, args.dense_arch, args.over_arch),
                "num_embeddings": "%s (%.1f GB fp32 tables)" % ("Criteo-1TB cardinalities capped at %d rows" % args.row_cap if args.config != "two_tower" else str(hashes),
                                                                sum(hashes) * args.embedding_dim * 4 / 1e9),
                "global_batch": B * world,
                "per_gpu_batch": B,
                "seq_len": args.pooling,
                "parallelism": f"{plan_info['rule']} embeddings ({plan_info['plan']} plan) over {world} GPU(s) + DDP dense"
                               + (f"; tables with <= {args.dp_rows} rows data-parallel" if world > 1 and args.dp_rows > 0 and args.sharding == "table_wise" else ""),
                "tables_per_rank": plan_info.get("tables_per_rank"),
                "transport": ("NVLink sparse plane (fused peer-memory kernels%s)" % (", CUDA-graph phases" if any(p._graphs for p in planes) else "")) if planes else "nccl / local",
                "overlap_sparse_dense": bool(args.overlap_sparse),
                "pipeline": "TrainPipelineSparseDist (e2e) / plain step (value)",
                "l2_policy": "inputs > L2: %d distinct batches, random rows of multi-GB tables (L2 126 MB)" % len(dev_batches),
                "dense_backend": dense_backend,
                "cuda_graphs": "dense sub-modules (fwd+bwd)" if args.cuda_graphs else "off",
                "cpu_binding": globals().get("_CPU_BINDING", "off"),
            },
            "clocks": clocks,
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": host_ms,
            "loss": float(loss.item()),
        }
        if e2e is not None:
            out["e2e"] = e2e
        if comm is not None:
            # BASELINE.json: "exposed all-to-all ms/step; pooled-emb all-to-all GB/s vs 900 GB/s". The input dist is hidden by the pipeline
            # (e2e) and inside the plain step it is part of `comm["input_dist_ms"]`.
            out["exposed_a2a_ms_per_step"] = comm["exposed_fwd_ms"] + comm["exposed_bwd_ms"]
            out["pooled_a2a_gbps"] = {"fwd_fused_with_lookup": comm["fwd_gbps"], "bwd_grad_push": comm["bwd_gbps"], "line_rate": 900.0,
                                      "frac_of_900": max(comm["fwd_gbps"], comm["bwd_gbps"]) / 900.0}
            out["comm"] = comm
        out.update(extra)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
