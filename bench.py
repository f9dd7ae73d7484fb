#!/usr/bin/env python
"""bench.py — headline benchmark of faabric_b200 (driver contract).

Headline (``--mode allreduce``, default): the reference's OWN all-reduce
benchmark workload (tests/dist/mpi/benchmarks/mpi_allreduce.cpp, "large"
payload): one pass = 214 MPI_Allreduce(MPI_INT, MPI_SUM) calls over the
ResNet-50 gradient tensors (25,583,592 int32 = 97.6 MiB).  A *step* is one
pass.  ``value`` is the whole-job algorithmic bandwidth  N * S / t  in GB/s
(S = bytes per rank per pass); ``busbw_GBps`` = 2(N-1)/N * S / t is reported
next to it against NVLink.  Device-timed with CUDA events, max over ranks.

Other modes (each prints one JSON line and appends to --out):
  sweep     MpiWorld allreduce bus GB/s 1 KB..1 GB, ours (per algo) vs NCCL
  alltoall  all-to-all bus GB/s 1 KB..64 MB per rank, ours vs NCCL
  snapshot  1 GB region diff+push at 1..50 % dirty (MB/s), vs CPU oracle rate; plus the runtime-level fork-join
  planner   1024-function fan-out / fan-in through the native planner (us)
  threads   THREADS fork-join of a 1 GiB device function memory through the runtime (ms)
  pingpong  MPI ping-pong RTT, 2 ranks in one worker and in two (CPU)
  hostcoll  host-buffer MPI collectives: reference algorithms vs shared memory (CPU)

Launch:  python bench.py --gpus 1          (single process)
         python -m torch.distributed.run --nnodes=1 --nproc-per-node N \
                --master-addr 127.0.0.1 --master-port P bench.py --gpus N
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl", "refcpu", "mpi-host", "mpi-device", "mpi-symmetric", "mpi-symmetric-nb"])
    ap.add_argument("--mode", default="allreduce",
                    choices=["allreduce", "sweep", "alltoall", "snapshot", "planner", "threads", "pingpong", "hostcoll"])
    ap.add_argument("--algo", default="tuned",
                    help="tuned = measure the algorithm policies in place and keep the fastest (allreduce mode)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--channels", type=int, default=8, help="lanes of --sync-mode lanes")
    ap.add_argument("--no-runtime-arm", action="store_true", help="snapshot mode: skip the THREADS fork-join through the runtime")
    ap.add_argument("--bind-numa", default="auto", choices=["auto", "on", "off"],
                    help="e2e: restrict the process to the CPUs of the GPU's NUMA node before allocating the pinned buffers (auto: multi-GPU runs only)")
    ap.add_argument("--no-mpi-api", action="store_true", help="skip the MPI C-API arm reported under 'mpi_api'")
    ap.add_argument("--sync-mode", default="grouped", choices=["grouped", "lanes"],
                    help="grouped = ONE fused kernel per step over all 214 tensors; lanes = one kernel per tensor")
    ap.add_argument("--no-nccl", action="store_true", help="skip the in-process graph-captured NCCL comparison")
    ap.add_argument("--e2e-chunks", type=int, default=8)
    ap.add_argument("--blocks", type=int, default=64, help="max CTAs per collective kernel (sweep modes)")
    ap.add_argument("--tuning", default="", help="JSON tuning table (default: profiles/tuning_N<gpus>.json)")
    ap.add_argument("--payload", default="large", choices=["large", "small"])
    ap.add_argument("--bucket-mb", type=float, default=25.0,
                    help="also report a DDP-style bucketed variant with this bucket size (0 = skip)")
    ap.add_argument("--out", default="")
    ap.add_argument("--max-bytes", type=int, default=1 << 30)
    ap.add_argument("--region-mb", type=int, default=1024)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="allreduce mode: after the timed steps write the all-reduced gradients of the last step "
                         "as DIR/grad_<i>.npy (float64, a fixed seeded sample of each tensor, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "allreduce" or args.impl != "ours"):
        ap.error("--dump-outputs needs --mode allreduce --impl ours")
    return args


def reference_arm(args):
    """The reference (faasm/faabric) is a conan/CMake C++ project; the offline
    pip install of /root/reference produces an empty 'UNKNOWN' package and its
    C++ build needs boost/protobuf/flatbuffers/nng/absl/spdlog/hiredis/zstd/
    catch2 + clang-17, none of which exist in this image (see DESIGN.md)."""
    print(json.dumps({
        "impl": "reference",
        "unavailable": "faabric is a conan+CMake C++ project: pip install of /root/reference yields an empty "
                       "package and its deps (boost, protobuf, flatbuffers, nng, absl, spdlog, hiredis, zstd) "
                       "are not installable offline",
    }))
    return 0


def refcpu_arm(args):
    """`refcpu`: the reference's OWN design - per-tensor MPI_Allreduce as
    reduce-to-rank-0 + broadcast over in-memory queues with malloc+memcpy per
    hop - run through this repo's native host path (C++, no GPU involved).
    World size = --gpus (min 2), ranks are executor threads of one worker."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from faabric_b200.models import resnet50_grad_sizes, small_sizes
    from faabric_b200.runtime import mpi_allreduce_bench

    sizes = resnet50_grad_sizes() if args.payload == "large" else small_sizes()
    n = max(args.gpus, 2)
    device = args.impl.startswith("mpi-")
    # refcpu = the reference's host algorithm; mpi-host = this repo's host path
    # (shared-memory slice-parallel all-reduce); mpi-{device,symmetric*} = HBM
    memory = args.impl[4:] if device else "host"
    res = mpi_allreduce_bench(sizes, n, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 3)),
                              memory=memory, host_algo="reference" if args.impl == "refcpu" else "shared")
    device = device and memory != "host"
    S = sum(sizes) * 4
    print(json.dumps({
        "metric": "mpi_allreduce_resnet50_grads_algbw_GBps",
        "impl": args.impl,
        "value": round(S / (res["ms_per_step"] * 1e-3) / 1e9, 4),
        "unit": "GB/s",
        "n_gpus": 0,
        "world_size": n,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(res["ms_per_step"], 3),
        "higher_is_better": True,
        "dtype": "int32",
        "data": "synthetic",
        "issue_ms_per_step": res.get("issue_ms_per_step"),
        "wait_ms_per_step": res.get("wait_ms_per_step"),
        "kernel_launches_per_step": res.get("kernel_launches_per_step"),
        "config": {"model": "resnet50-gradients", "tensors": len(sizes), "bytes": S,
                   "path": f"MPI C API ({args.impl[4:]} memory), one fused kernel per MPI call" if device
                   else "host memory, reduce-to-root + broadcast over in-memory queues"},
    }), flush=True)
    return 0


def mode_pingpong(args):
    """BASELINE config 1: MPI ping-pong, world_size=2, CPU only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from faabric_b200.runtime import cpu_pingpong_bench

    local = cpu_pingpong_bench(sizes=(8, 1024, 65536), n_workers=1)
    tcp = cpu_pingpong_bench(sizes=(8, 1024, 65536), n_workers=2)
    print(json.dumps({
        "metric": "mpi_pingpong_rtt_us_8B",
        "value": local[0]["rtt_us"],
        "unit": "us",
        "higher_is_better": False,
        "n_gpus": 0,
        "world_size": 2,
        "details": {"same_worker_queue": local, "two_workers_tcp": tcp},
    }), flush=True)
    return 0


def mode_hostcoll(args):
    """Host-buffer MPI collectives inside one worker: reference algorithms vs
    the shared-memory path (CPU only; table in profiles/README.md)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from faabric_b200.runtime import host_collectives_bench

    cells = host_collectives_bench(repeats=max(1, min(args.steps, 5)))
    key = "shared-8-8388608"
    ref = "reference-8-8388608"
    print(json.dumps({
        "metric": "mpi_host_allreduce_8MiB_8ranks_us",
        "value": cells[key]["allreduce_us"],
        "unit": "us",
        "higher_is_better": False,
        "n_gpus": 0,
        "reference_algorithm_us": cells[ref]["allreduce_us"],
        "details": cells,
    }), flush=True)
    return 0


# ----------------------------------------------------------------------------
# distributed plumbing
# ----------------------------------------------------------------------------
class Dist:
    def __init__(self, want_gpus: int):
        import torch

        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.multi = self.world > 1
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device")
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        self.pg = None
        if self.multi:
            import torch.distributed as dist

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.device)
            self.pg = dist
        if want_gpus != self.world and self.rank == 0 and self.world > 1:
            print(f"[bench] --gpus {want_gpus} but WORLD_SIZE={self.world}; using WORLD_SIZE", file=sys.stderr)

    def barrier(self):
        if self.pg is not None:
            self.pg.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.pg is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.device)
        self.pg.all_reduce(t, op=self.pg.ReduceOp.MAX)
        return float(t.item())

    def make_comm(self, **cfg):
        from faabric_b200.parallel import LocalGroup, init_from_env

        if self.multi:
            return init_from_env(**cfg), None
        g = LocalGroup(1, devices=[self.local], **cfg)
        return g.comms[0], g

    def close(self):
        if self.pg is not None:
            self.pg.destroy_process_group()


def timed(dist: Dist, fn, steps: int, warmup: int):
    """W untimed warm-ups, then exactly `steps` calls bracketed by a barrier +
    synchronize on both sides and CUDA events; returns max-over-ranks ms/step."""
    torch = dist.torch
    for _ in range(warmup):
        fn()
    dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    dist.barrier()
    return dist.max_over_ranks(ms)


def load_tuning(comm, args, dist):
    """Apply the measured algorithm table for this world size, if present."""
    path = Path(args.tuning) if args.tuning else ROOT / "profiles" / f"tuning_N{dist.world}.json"
    if not path.exists():
        return None
    try:
        if path.suffix != ".json":  # native text format (faabric_b200.parallel.autotune)
            comm.load_tuning(path)
            return str(path)
        t = json.loads(path.read_text())
        comm.set_allreduce_table([(e["max_bytes"], e["algo"]) for e in t["allreduce"]])
        return str(path)
    except Exception as e:  # noqa: BLE001
        print(f"[bench] tuning file {path} ignored: {e}", file=sys.stderr)
        return None


def dump_outputs(out_dir, views, budget_bytes=48 << 20, seed=0):
    """Write each tensor of `views` as float64 (exact for int32) to
    out_dir/grad_<i>.npy.  When the whole set exceeds `budget_bytes`, every
    tensor is cut to the same fraction of its elements, picked by a fixed seed
    and kept in index order, so that runs of two builds compare element for element."""
    import numpy as np
    import torch

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    frac = min(1.0, budget_bytes / 8 / sum(v.numel() for v in views))
    gen = torch.Generator().manual_seed(seed)
    for i, v in enumerate(views):
        n = v.numel()
        k = max(1, int(n * frac))
        if k < n:
            v = v[torch.randperm(n, generator=gen)[:k].sort().values.to(v.device)]
        np.save(out / f"grad_{i:03d}.npy", v.to(torch.float64).cpu().numpy())


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text())
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "fallback": True}


# ----------------------------------------------------------------------------
# headline: ResNet-50 gradient all-reduce pass
# ----------------------------------------------------------------------------
def mode_allreduce(args, dist: Dist):
    import torch
    from faabric_b200.models import GradientSync, resnet50_grad_sizes, small_sizes
    from faabric_b200.utils import ClockSampler

    sizes = resnet50_grad_sizes() if args.payload == "large" else small_sizes()
    n = dist.world
    S = sum(sizes) * 4
    result = {}

    def nccl_graph_ms():
        """The same 214-call loop over NCCL, captured ONCE into a CUDA graph
        and replayed (no Python / c10d overhead per call): the fair baseline."""
        bufs = [torch.zeros(s_, dtype=torch.int32, device=dist.device) for s_ in sizes]
        side = torch.cuda.Stream(device=dist.device)
        with torch.cuda.stream(side):
            for b in bufs:
                dist.pg.all_reduce(b)
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for b in bufs:
                dist.pg.all_reduce(b)
        ms_ = timed(dist, g.replay, args.steps, args.warmup)
        del g
        return ms_

    if args.impl == "nccl":
        if not dist.multi:
            raise SystemExit("--impl nccl needs >1 rank")
        sampler = ClockSampler(gpu_index=dist.local).start() if dist.rank == 0 else None
        ms = nccl_graph_ms()
        clocks = sampler.stop() if sampler else {}
        launches = 0
        e2e = None
        cfg_extra = {"library": "NCCL all_reduce x214, CUDA-graph captured (baseline, not the product)"}
    else:
        grouped = args.sync_mode == "grouped"
        comm, group = dist.make_comm(heapBytes=(512 << 20), stageBytes=(16 << 20),
                                     channels=1 if grouped else args.channels)
        load_tuning(comm, args, dist)
        sync = GradientSync(comm, sizes, dtype=torch.int32, algo=args.algo, use_graph=not args.no_graph,
                            channels=args.channels, mode=args.sync_mode)
        # deterministic non-trivial contents
        sync.send.copy_(torch.arange(sync.send.numel(), device=dist.device, dtype=torch.int32) % 1000 + dist.rank)
        torch.cuda.synchronize()
        # ---- correctness check before timing: EVERY tensor against the closed form
        sync.step()
        torch.cuda.synchronize()
        pos = torch.arange(sync.send.numel(), device=dist.device, dtype=torch.int64) % 1000
        exp_flat = (pos * n + n * (n - 1) // 2).to(torch.int32)
        for o, sz in zip(sync.offsets, sync.sizes):
            if not torch.equal(sync.recv[o:o + sz], exp_flat[o:o + sz]):
                raise SystemExit(f"all-reduce result mismatch in tensor at offset {o}")
        del pos
        comm.stats(reset=True)
        sampler = ClockSampler(gpu_index=dist.local).start() if dist.rank == 0 else None
        ms = timed(dist, sync.step, args.steps, args.warmup)
        clocks = sampler.stop() if sampler else {}
        if args.dump_outputs and dist.rank == 0:
            dump_outputs(args.dump_outputs, sync.recv_views)
        launches = sync.launches_per_step * args.steps
        err = comm.check_error()
        if err:
            raise SystemExit(f"device watchdog error {err}")
        # ---- end to end through the public API:
        # pinned host -> H2D -> all-reduce -> D2H of the FULL result into pinned host memory
        from faabric_b200.utils import bind_process_near_gpu
        numa_cpus = bind_process_near_gpu(dist.local) if (args.bind_numa == "on" or (args.bind_numa == "auto" and dist.multi)) else []
        host = torch.empty(sync.total_padded, dtype=torch.int32).pin_memory()
        host.copy_((torch.arange(sync.total_padded, dtype=torch.int32) % 1000) + dist.rank)
        out_host = torch.empty(sync.total_padded, dtype=torch.int32).pin_memory()
        for _ in range(max(3, args.warmup)):
            sync.step_from_host(host, pipeline=args.e2e_chunks, out_host=out_host)
        dist.barrier()
        t0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            res = sync.step_from_host(host, pipeline=args.e2e_chunks, out_host=out_host)
        e1.record()
        torch.cuda.synchronize()
        e2e_ms = dist.max_over_ranks(e0.elapsed_time(e1) / args.steps)
        wall_ms = dist.max_over_ranks((time.perf_counter() - t0) * 1000 / args.steps)
        e2e_ms = max(e2e_ms, wall_ms)  # host-synchronous steps: the wall clock governs
        if grouped:
            exp_host = exp_flat.cpu()
            for o, sz in list(zip(sync.offsets, sync.sizes))[:: max(1, len(sync.sizes) // 16)]:
                if not torch.equal(res[o:o + sz], exp_host[o:o + sz]):
                    raise SystemExit(f"e2e result mismatch in tensor at offset {o}")
        else:
            if int(res[0]) != n * (n - 1) // 2:
                raise SystemExit("e2e digest mismatch")
        e2e = {
            "value": round(n * S / (e2e_ms * 1e-3) / 1e9, 3),
            "unit": "GB/s",
            "ms_per_step": round(e2e_ms, 4),
            "h2d_bytes_per_step": sync.h2d_bytes_per_step,
            "d2h_bytes_per_step": sync.d2h_bytes_per_step,
            "pipeline_chunks": args.e2e_chunks,
            "numa_bound_cpus": len(numa_cpus),
            "result_checked_on_host": True,
        }
        del exp_flat
        # ---- fair library baseline, same process, same box
        nccl_ms = None
        if dist.multi and not args.no_nccl:
            try:
                nccl_ms = nccl_graph_ms()
            except Exception as ex:  # noqa: BLE001
                print(f"[bench] NCCL comparison skipped: {ex}", file=sys.stderr)
        st = comm.stats()
        cfg_extra = {
            "sync_mode": args.sync_mode,
            "backing": comm.backing,
            "nvls": comm.has_multicast,
            "cuda_graph": (not args.no_graph) and not grouped,
            "channels": 1 if grouped else args.channels,
            "algo": "two-shot peer-memory, grouped" if grouped else args.algo,
            "tuned_policy": sync.policy_name,
            "tuned_policy_ms": sync.policy_timings,
            "algo_mix": {k: v for k, v in st.items() if k.startswith("algo_") and v},
            "launches_per_step": sync.launches_per_step,
        }
        if nccl_ms is not None:
            result["nccl_graph_ms"] = nccl_ms
        result["_keep"] = (sync, comm, group)

    algbw = n * S / (ms * 1e-3) / 1e9
    busbw = (2 * (n - 1) / n) * S / (ms * 1e-3) / 1e9 if n > 1 else 0.0
    pk = peaks()
    out = {
        "metric": "mpi_allreduce_resnet50_grads_algbw_GBps",
        "value": round(algbw, 3),
        "unit": "GB/s",
        "n_gpus": n,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(ms, 4),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "int32",
        "data": "synthetic",
        "impl": args.impl,
        "busbw_GBps": round(busbw, 3),
        "busbw_frac_of_nvlink_770": round(busbw / 770.0, 4) if n > 1 else None,
        "us_per_allreduce": round(ms * 1000 / len(sizes), 3),
        "gpu_launches": launches,
        "clocks": clocks,
        "config": {
            "model": "resnet50-gradients (reference mpi_bench 'large' payload)" if args.payload == "large"
            else "1000 x 8-int messages (reference 'small' payload)",
            "tensors": len(sizes),
            "elements": sum(sizes),
            "bytes_per_rank_per_step": S,
            "global_batch": None,
            "seq_len": None,
            "parallelism": f"dp{n}",
            "op": "MPI_Allreduce(MPI_INT, MPI_SUM) per tensor (214 independent results)",
            "l2": "inputs+outputs per step = 2 x 97.6 MiB > 126 MB L2 (no flush needed)",
            "timing": "CUDA events, barrier+sync both sides, max over ranks",
            "value_definition": "N*S/t (whole-job bytes all-reduced per second); busbw=2(N-1)/N*S/t",
            "measured_hbm_gbs": pk.get("hbm_gbs"),
            **cfg_extra,
        },
    }
    if e2e is not None:
        out["e2e"] = e2e
    if result.get("nccl_graph_ms"):
        out["nccl_graph_ms_per_step"] = round(result["nccl_graph_ms"], 4)
        out["vs_nccl"] = round(result["nccl_graph_ms"] / ms, 3)
    return out, result


# ----------------------------------------------------------------------------
# sweep: allreduce bus bandwidth by size, ours (each algo) vs NCCL
# ----------------------------------------------------------------------------
def _sizes(lo, hi):
    s = lo
    out = []
    while s <= hi:
        out.append(s)
        s *= 4
    if out[-1] != hi:
        out.append(hi)
    return out


def mode_sweep(args, dist: Dist):
    import torch

    n = dist.world
    maxb = args.max_bytes
    comm, group = dist.make_comm(heapBytes=2 * maxb + (64 << 20), stageBytes=(16 << 20), maxBlocks=args.blocks, channels=1)
    send = comm.empty(maxb // 4, torch.float32)
    recv = comm.empty(maxb // 4, torch.float32)
    send.fill_(1.0)
    rows = []
    algos = ["ll", "oneshot", "twoshot"] + (["nvls"] if comm.has_multicast else []) + ["auto"]
    for nbytes in _sizes(1024, maxb):
        numel = nbytes // 4
        row = {"bytes": nbytes}
        iters = 200 if nbytes <= (1 << 20) else (40 if nbytes <= (64 << 20) else 10)
        for algo in algos:
            if algo == "ll" and nbytes > 65536:
                continue
            if algo == "oneshot" and nbytes > (16 << 20):
                continue
            s, r = send[:numel], recv[:numel]
            try:
                ms = timed(dist, lambda: comm.all_reduce(s, r, algo=algo), iters, 5)
            except Exception as e:  # noqa: BLE001
                row[algo] = f"error: {e}"
                continue
            row[algo + "_us"] = round(ms * 1000, 2)
            row[algo + "_busbw"] = round((2 * (n - 1) / n) * nbytes / (ms * 1e-3) / 1e9, 2) if n > 1 else round(nbytes / (ms * 1e-3) / 1e9, 2)
            if algo == "auto":
                row["auto_pick"] = comm.last_algo
        if dist.multi:
            t = torch.ones(numel, dtype=torch.float32, device=dist.device)
            ms = timed(dist, lambda: dist.pg.all_reduce(t), iters, 5)
            row["nccl_us"] = round(ms * 1000, 2)
            row["nccl_busbw"] = round((2 * (n - 1) / n) * nbytes / (ms * 1e-3) / 1e9, 2)
        rows.append(row)
        if dist.rank == 0:
            print("[sweep]", json.dumps(row), file=sys.stderr, flush=True)
    err = comm.check_error()
    # measured selection table: fastest algorithm per size bucket
    table = []
    from faabric_b200.parallel import autotune

    merged = autotune.json_table_from_rows(rows)
    if dist.rank == 0:
        tp = Path("gpurun_out") / f"tuning_N{n}.json"
        tp.parent.mkdir(exist_ok=True)
        tp.write_text(json.dumps({"n_gpus": n, "allreduce": merged, "source": "bench.py --mode sweep", "rows": rows}, indent=1))
        # same table in the format FAABRIC_TUNING_FILE takes
        autotune.write_tuning_file(tp.with_suffix(".txt"), autotune.table_from_rows(rows), comment=f"bench.py --mode sweep, {n} GPUs, fp32")
    best = max((r.get("auto_busbw", 0) for r in rows), default=0)
    out = {
        "metric": "mpi_allreduce_busbw_sweep_GBps",
        "value": best,
        "unit": "GB/s (peak auto bus bandwidth in sweep)",
        "n_gpus": n,
        "dtype": "fp32",
        "data": "synthetic",
        "higher_is_better": True,
        "device_error": err,
        "backing": comm.backing,
        "nvls": comm.has_multicast,
        "rows": rows,
        "tuning_table": merged,
        "roofline": "NVLink5 770 GB/s measured per direction per GPU (900 nominal)",
    }
    return out, {"_keep": (comm, group, send, recv)}


def mode_alltoall(args, dist: Dist):
    import torch

    n = dist.world
    max_per_rank = min(args.max_bytes, 64 << 20)
    comm, group = dist.make_comm(heapBytes=2 * max_per_rank * n + (64 << 20), stageBytes=(16 << 20), maxBlocks=args.blocks, channels=1)
    send = comm.empty(max_per_rank * n // 4, torch.float32)
    recv = comm.empty(max_per_rank * n // 4, torch.float32)
    send.fill_(2.0)
    rows = []
    for per in _sizes(1024, max_per_rank):
        numel = per * n // 4
        iters = 200 if per <= (1 << 20) else 30
        s, r = send[:numel], recv[:numel]
        ms = timed(dist, lambda: comm.all_to_all(s, r), iters, 5)
        total = per * n
        row = {
            "bytes_per_rank_pair": per,
            "ours_us": round(ms * 1000, 2),
            "ours_busbw": round(((n - 1) / n) * total / (ms * 1e-3) / 1e9, 2) if n > 1 else round(total / (ms * 1e-3) / 1e9, 2),
        }
        if dist.multi:
            a = torch.ones(numel, dtype=torch.float32, device=dist.device)
            b = torch.empty_like(a)
            ms2 = timed(dist, lambda: dist.pg.all_to_all_single(b, a), iters, 5)
            row["nccl_us"] = round(ms2 * 1000, 2)
            row["nccl_busbw"] = round(((n - 1) / n) * total / (ms2 * 1e-3) / 1e9, 2)
        rows.append(row)
        if dist.rank == 0:
            print("[alltoall]", json.dumps(row), file=sys.stderr, flush=True)
    out = {
        "metric": "mpi_alltoall_busbw_sweep_GBps",
        "value": max(r["ours_busbw"] for r in rows),
        "unit": "GB/s (peak)",
        "n_gpus": n,
        "dtype": "fp32",
        "data": "synthetic",
        "higher_is_better": True,
        "device_error": comm.check_error(),
        "rows": rows,
    }
    return out, {"_keep": (comm, group, send, recv)}


def mode_snapshot(args, dist: Dist):
    """1 GB region: every non-main GPU diffs its memory against its base image
    and pushes the merged bytes straight into the main GPU's image."""
    import numpy as np
    import torch
    from faabric_b200.ops import snapshot as snap

    n = dist.world
    size = args.region_mb << 20
    comm, group = dist.make_comm(heapBytes=size + (64 << 20), stageBytes=(16 << 20))
    main_img = comm.empty(size, torch.uint8)  # symmetric: rank 0's copy is the main image
    main_img.zero_()
    base = torch.zeros(size, dtype=torch.uint8, device=dist.device)
    mem = torch.zeros(size, dtype=torch.uint8, device=dist.device)
    regs = snap.prepare_regions([], size, dist.device)
    # peer-mapped pointer of rank 0's image
    dst_ptr = comm._lib.fb_comm_heap_ptr(comm._h, comm.heap_offset(main_img), 0)
    n_pages = size // 4096
    rows = []
    gen = torch.Generator(device=dist.device).manual_seed(1234 + dist.rank)
    for pct in (1, 5, 10, 25, 50):
        n_dirty = n_pages * pct // 100
        perm = torch.randperm(n_pages, generator=gen, device=dist.device)[:n_dirty]
        mem.copy_(base)
        mem.view(n_pages, 4096)[perm] = torch.randint(
            1, 255, (n_dirty, 4096), dtype=torch.uint8, device=dist.device, generator=gen
        )
        flags = torch.zeros(n_pages, dtype=torch.uint8, device=dist.device)
        flags[perm] = 1
        stats = torch.zeros(2, dtype=torch.int64, device=dist.device)
        torch.cuda.synchronize()
        row = {"dirty_pct": pct, "dirty_bytes": n_dirty * 4096}
        for label, dirty in (("scan_all", None), ("tracked", flags)):
            def run():
                stats.zero_()
                snap.diff_push(mem, base, dst_ptr, regs, dirty_pages=dirty, stats=stats)
            ms = timed(dist, run, max(3, args.steps // 2), 3)
            row[label + "_ms"] = round(ms, 4)
            row[label + "_region_GBps"] = round(size / (ms * 1e-3) / 1e9, 1)
            row[label + "_dirty_GBps"] = round(n_dirty * 4096 / (ms * 1e-3) / 1e9, 1)
        row["diff_bytes"] = int(stats[0].item())
        # roofline: max(2*region/HBM (every rank scans its own copy),
        #               incast into the main image: (N-1)*dirty / NVLink ingress of ONE GPU)
        pk = peaks()
        t_scan = 2 * size / (pk.get("hbm_gbs", 6650.0) * 1e9)
        if n > 1:
            t_push = (n - 1) * (n_dirty * 4096) / 770e9
        else:
            t_push = (n_dirty * 4096) / (pk.get("hbm_gbs", 6650.0) * 1e9)
        row["roofline_terms_ms"] = {"scan": round(t_scan * 1e3, 4), "incast_push": round(t_push * 1e3, 4)}
        row["roofline_ms_scan_all"] = round(max(t_scan, t_push) * 1e3, 4)
        row["frac_of_roofline_scan_all"] = round(max(t_scan, t_push) * 1e3 / row["scan_all_ms"], 3)
        rows.append(row)
        if dist.rank == 0:
            print("[snapshot]", json.dumps(row), file=sys.stderr, flush=True)
    # CPU oracle rate (reference semantics: 128-B chunk memcmp + byte runs + memcpy)
    cpu = {}
    if dist.rank == 0:
        a = np.zeros(64 << 20, dtype=np.uint8)
        b = a.copy()
        b[:: 4096 * 10] = 1
        t0 = time.perf_counter()
        d = np.nonzero(a.reshape(-1, 128) != b.reshape(-1, 128))[0]
        cpu["numpy_compare_GBps"] = round(len(a) / (time.perf_counter() - t0) / 1e9, 2)
        cpu["chunks"] = int(len(d))
    out = {
        "metric": "snapshot_diff_push_region_MBps",
        "value": round(rows[0]["scan_all_region_GBps"] * 1000, 1),
        "unit": "MB/s of region processed per GPU (1% dirty, scan-all mode)",
        "n_gpus": n,
        "region_bytes": size,
        "data": "synthetic",
        "higher_is_better": True,
        "rows": rows,
        "cpu_oracle": cpu,
        "note": "every rank pushes into rank 0's image over NVLink (rank 0 pushes locally)",
    }
    # The same kernels where the runtime uses them: a THREADS fork-join through planner, scheduler,
    # DeviceExecutor and SnapshotRegistry (one thread per virtual GPU host, 1 GiB function memory)
    if dist.rank == 0 and not args.no_runtime_arm:
        try:
            from faabric_b200.runtime import threads_forkjoin_bench

            fj = threads_forkjoin_bench("device", hosts=max(n, 2), iters=10, warmup=3)
            out["runtime_forkjoin"] = {k: fj.get(k) for k in ("hosts", "gpus", "mem_bytes", "dirty_pct", "ms_median", "ms_min",
                                                                "diff_push_kernels", "verified")}
        except Exception as e:  # the kernel rows never depend on this arm
            out["runtime_forkjoin"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    return out, {"_keep": (comm, group, main_img)}


def mode_planner(args, dist: Dist):
    from faabric_b200.runtime import planner_fanout_bench

    res = planner_fanout_bench(n_functions=1024, n_hosts=8, iters=max(args.steps, 5), warmup=max(args.warmup, 2))
    ref = planner_fanout_bench(n_functions=1024, n_hosts=8, iters=max(args.steps, 5), warmup=max(args.warmup, 2), mode="refcpu")
    out = {
        "metric": "planner_fanout_fanin_1024_us",
        "value": res["us_per_batch_median"],
        "unit": "us",
        "higher_is_better": False,
        "n_gpus": 0,
        "refcpu_us": ref["us_per_batch_median"],
        "vs_refcpu": round(ref["us_per_batch_median"] / res["us_per_batch_median"], 2),
        "details": res,
        "refcpu_details": ref,
        "note": "refcpu = the reference's design (every request/result encoded + sent over a loopback socket + decoded), "
                "run by this repo's planner on the same box",
    }
    return out, {}


def mode_threads(args, dist: Dist):
    """THREADS fork-join through the whole runtime on device memory, against the
    reference's host-memory design (mprotect tracking + byte diffs) on the same box."""
    from faabric_b200.runtime import threads_forkjoin_bench

    hosts = args.gpus if args.gpus > 1 else 2
    dev = threads_forkjoin_bench("device", hosts=hosts, iters=max(args.steps, 5), warmup=max(args.warmup, 2))
    ref = threads_forkjoin_bench("host", hosts=hosts, iters=5, warmup=1)
    out = {
        "metric": "threads_forkjoin_1GiB_ms",
        "value": dev.get("ms_median"),
        "unit": "ms",
        "higher_is_better": False,
        "n_gpus": dev.get("gpus"),
        "refcpu_ms": ref.get("ms_median"),
        "vs_refcpu": round(ref["ms_median"] / dev["ms_median"], 2) if dev.get("ms_median") else None,
        "details": dev,
        "refcpu_details": ref,
        "note": "executeThreads() wall time, one thread per virtual GPU host, 1% of a 1 GiB function memory dirtied per join; "
                "refcpu = host memory, mprotect dirty tracking, byte diffs through the snapshot server",
    }
    return out, {}


def mpi_api_arm(n: int, steps: int, warmup: int) -> dict:
    """Runs `bench.py --impl mpi-symmetric-nb` in a child (its own worker process with n rank threads)."""
    import subprocess

    env = {k: v for k, v in os.environ.items()
           if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "MASTER_ADDR",
                        "MASTER_PORT", "TORCHELASTIC_RUN_ID")}
    try:
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "mpi-symmetric-nb", "--gpus", str(n),
                            "--steps", str(steps), "--warmup", str(warmup)], capture_output=True, text=True, timeout=300, env=env)
        res = json.loads(r.stdout.strip().splitlines()[-1])
        return {"impl": "MPI_Iallreduce x214 + MPI_Waitall (C API, symmetric device memory)", "world_size": res["world_size"],
                "ms_per_step": res["ms_per_step"], "us_per_allreduce": round(res["ms_per_step"] * 1000 / res["config"]["tensors"], 3),
                "issue_ms_per_step": res.get("issue_ms_per_step"), "wait_ms_per_step": res.get("wait_ms_per_step"),
                "kernel_launches_per_step": res.get("kernel_launches_per_step")}
    except Exception as e:  # the headline never depends on this arm
        return {"error": f"{type(e).__name__}: {str(e)[:200]}"}


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    if args.impl == "refcpu" or args.impl.startswith("mpi-"):
        return refcpu_arm(args)
    if args.mode == "pingpong":
        return mode_pingpong(args)
    if args.mode == "hostcoll":
        return mode_hostcoll(args)
    if args.mode in ("planner", "threads"):
        # one process drives everything: no process group needed
        if int(os.environ.get("RANK", "0")) == 0:
            out, _ = (mode_planner if args.mode == "planner" else mode_threads)(args, None)
            print(json.dumps(out), flush=True)
        return 0
    dist = Dist(args.gpus)
    fn = {
        "allreduce": mode_allreduce,
        "sweep": mode_sweep,
        "alltoall": mode_alltoall,
        "snapshot": mode_snapshot,
        "planner": mode_planner,
    }[args.mode]
    out, keep = fn(args, dist)
    if args.mode == "allreduce" and args.impl == "ours" and not args.no_mpi_api:
        # the same 214 reductions through the product's MPI C API (MPI_Iallreduce x214 + MPI_Waitall on
        # symmetric device memory, ranks = executor threads of one worker process), reported next to the headline
        keep = None
        dist.torch.cuda.synchronize()
        if dist.rank == 0:
            out["mpi_api"] = mpi_api_arm(max(dist.world, 2), args.steps, args.warmup)
    if dist.rank == 0:
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")
    dist.barrier()
    del keep
    dist.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
