"""Headline benchmark: MNIST-MLP steps/sec of the parameter-server engine, whole box, device-timed.

    python bench.py --gpus 1 --steps 2000 --warmup 50
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Topology (BASELINE.json configs): N = 1 -> 1 ps + 1 worker sharing the GPU (one process);
N >= 2 -> rank 0 is the dedicated ps GPU, ranks 1..N-1 are workers (N = 8 -> "1 ps + 7 workers").
Model/config: the reference's live model (784-100-10 "book" MLP, batch 32 per worker, Adam lr 1e-4,
asynchronous per-push apply on the ps) with synthetic 28x28 data and random-init weights.

Numbers in the JSON line (all: max over ranks, throughput = workers x K / max elapsed):
  value    : K steps per worker, inputs read from a device-resident 55 000-image dataset (172 MB > L2) — with the
             fused engine ONE kernel launch whose TMA loads take the batch rows straight out of the dataset —
             timed with CUDA events on the worker's compute stream; the region ends with a stream-ordered wait for
             the ps acknowledgement of the last push, so every step's pull, math, push and optimizer apply is inside.
  e2e      : the same K steps through the public API (`Worker.run_steps`): native next_batch out of the loader's
             epoch-shuffled pinned buffer (TF DataSet semantics: rows are shuffled physically once per epoch — here by
             background threads — and a batch is a contiguous slice), H2D copy of every batch from that pinned memory,
             step kernels, 16-byte result read back per step; wall clock between device synchronisations, closed by the
             ps acknowledgement of the last push. `input_feed` in the e2e object says which path fed the timed steps.
  parity   : the reference's worker semantics — one step at a time per worker (`--lanes 1`), host-fed — and the same
             with `--strict_steps` (the next pull waits for the acknowledgement of the previous push).
  roofline : achieved fraction of the NVLink / HBM / tensor-core rooflines from MEASURED_PEAKS.json.

--dump-outputs DIR: after the device-timed region, the chief worker writes what its last step returned (`loss.npy`,
`correct.npy`) and the variables on the ps shards (`var_<name>.npy`, "/" in a name becomes "__") as float32. Data and
initial variables are seeded, so two builds run with the same arguments start from identical inputs; with more than
one step in flight (`--lanes`) the staleness of each pull depends on timing, so compare with a tolerance.

Steps in flight: a worker keeps `--lanes` (default 12, the CLI's default too) steps in flight on its GPU — bounded-
staleness asynchronous SGD: every step still pulls, computes, pushes and is applied on the ps individually.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import torch

REFERENCE_UNAVAILABLE = (
    "reference needs TensorFlow 1.x (tf.contrib, tf.app.flags, tf.train.Server); no tensorflow wheel in "
    "/opt/wheelhouse, none for Python 3.12, no network; /root/reference has no setup.py/pyproject so "
    "`pip install --target baseline/_ref /root/reference` fails with 'not installable'"
)
NVLINK_GBS = 770.0   # measured peer-copy bandwidth per direction per GPU (profiling recipe)
DUMP_MAX_BYTES = 60 << 20   # --dump-outputs: array data in all (the .npy headers stay well inside 64 MB)


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2000)
    p.add_argument("--warmup", type=int, default=50)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--model", default="book")
    p.add_argument("--hidden_units", type=int, default=100)
    p.add_argument("--batch_size", type=int, default=32)
    p.add_argument("--optimizer", choices=["adam", "sgd"], default="adam")
    p.add_argument("--learning_rate", type=float, default=1e-4)
    p.add_argument("--dtype", choices=["fp32", "bf16"], default="fp32")
    p.add_argument("--push_mode", choices=["mailbox", "atomic"], default="mailbox")
    p.add_argument("--apply_mode", choices=["per_push", "merged"], default="per_push")
    p.add_argument("--num_ps", type=int, default=1)
    p.add_argument("--sharding", choices=["round_robin", "byte_balanced", "row_split"], default="round_robin")
    p.add_argument("--engine", choices=["auto", "fused", "graph"], default="auto")
    p.add_argument("--nslots", type=int, default=0, help="mailbox slots per worker (0 = max(4 x lanes, 8))")
    p.add_argument("--lanes", type=int, default=12,
                   help="steps of one worker in flight on its GPU at once (async SGD; must be <= nslots)")
    p.add_argument("--strict_steps", action="store_true")
    p.add_argument("--graph_steps", type=int, default=0,
                   help="graph engine: steps per CUDA-graph launch in the native loops (0 = min(lanes, 4))")
    p.add_argument("--ps_row_blocks", type=int, default=4)
    p.add_argument("--skip_e2e", action="store_true")
    p.add_argument("--skip_parity", action="store_true")
    p.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                   help="after the device-timed steps, write the result of their last step and the variables it left "
                        "on the ps as DIR/<name>.npy (float32), to compare two builds output for output")
    return p.parse_args(argv)


def engine_config(args, backend: str = "cuda"):
    """Same derivation as `dist_mnist_b200.cli.engine_config_from_args` (tests compare the two)."""
    from dist_mnist_b200.parallel.config import EngineConfig

    lanes = max(1, args.lanes)
    return EngineConfig(backend=backend, dtype=args.dtype, nslots=args.nslots or max(4 * lanes, 8), apply_mode=args.apply_mode,
                        push_mode=args.push_mode, sharding=args.sharding, lanes=lanes,
                        graph_steps=args.graph_steps or next(u for u in (4, 3, 2, 1) if lanes % u == 0),
                        pipeline_slots=max(4, 2 * lanes),
                        engine=args.engine, strict_steps=args.strict_steps, ps_row_blocks=args.ps_row_blocks)


def _usable_cores():
    try:
        from dist_mnist_b200.parallel.worker import usable_cores
        return usable_cores()
    except Exception:
        return None


def load_peaks() -> dict:
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]), "source": "MEASURED_PEAKS.json"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback (profiling recipe)"}


def main(argv=None) -> int:
    args = parse_args(argv)
    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable": REFERENCE_UNAVAILABLE}))
        return 0

    # Hang watchdog: a healthy run takes seconds to a couple of minutes (the first `import torch` on a fresh box
    # included). If something deadlocks, dump every Python thread's stack to stderr and exit instead of sitting in the
    # caller's timeout without a trace. DM_BENCH_WATCHDOG_S=0 switches it off.
    import faulthandler
    watchdog_s = int(os.environ.get("DM_BENCH_WATCHDOG_S", "1500"))
    if watchdog_s > 0:
        faulthandler.dump_traceback_later(watchdog_s, exit=True)

    import torch.distributed as dist

    from dist_mnist_b200 import _native as N
    from dist_mnist_b200.cluster import ClusterSpec, Rendezvous
    from dist_mnist_b200.models import mlp
    from dist_mnist_b200.parallel.config import OptimizerConfig
    from dist_mnist_b200.parallel.ps import ParameterServer
    from dist_mnist_b200.parallel.worker import Worker
    from dist_mnist_b200.session import InProcessCluster
    from dist_mnist_b200.utils import data as data_utils
    from dist_mnist_b200.utils.metrics import ClockSampler, StreamTimer

    if not torch.cuda.is_available():
        print(json.dumps({"error": "bench.py needs a CUDA device (B200); none visible"}))
        return 1
    N.lib()  # fail loudly if the native library is missing: there is no eager fallback for the hot path

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = args.gpus
    if world > 1 and world != n_gpus:
        raise SystemExit(f"--gpus {n_gpus} but WORLD_SIZE={world}")
    if world == 1 and n_gpus != 1:
        raise SystemExit("for --gpus N > 1 launch with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        # NCCL builds its communicator lazily inside the first collective (hundreds of milliseconds): do that now, not
        # inside the barrier that precedes the first timed region (the NVLink sublinks would fall asleep meanwhile)
        dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    spec = mlp.get_model(args.model, args.hidden_units)
    opt = OptimizerConfig(args.optimizer, args.learning_rate)
    cfg = engine_config(args)
    cfg.validate(opt)
    engine = cfg.resolve_engine(spec, args.batch_size)
    K, W, B = args.steps, max(args.warmup, 3), args.batch_size

    # ---------------- data (allocated before any persistent PS kernel exists on this GPU) ----------------
    ds = data_utils.synthetic_mnist(data_utils.TRAIN_SIZE, seed=0)
    is_worker_rank = world == 1 or rank >= args.num_ps
    dev_x = dev_y = None
    if is_worker_rank:
        dev = torch.device("cuda", local_rank)
        tdtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
        dev_x = ds.images.to(tdtype).to(dev).contiguous()      # 55000 x 784: 172 MB fp32 (> 126 MB L2)
        dev_y = ds.labels.to(dev).contiguous()
        torch.cuda.synchronize()

    # ---------------- bring-up ----------------
    ps_list, worker, inproc = [], None, None
    loaders = {}

    def make_loader(w):
        loaders["l"] = w.make_loader(ds.images, ds.labels, seed=rank)

    if world == 1:
        inproc = InProcessCluster(spec, opt, cfg, batch_size=B, num_ps=args.num_ps, device=local_rank, seed=0,
                                  setup_hook=make_loader)
        ps_list, worker = inproc.ps, inproc.worker
        n_workers = 1
    else:
        num_ps = args.num_ps
        n_workers = world - num_ps
        if n_workers < 1:
            raise SystemExit("need at least one worker rank")
        addr = os.environ.get("MASTER_ADDR", "127.0.0.1")
        port = int(os.environ.get("MASTER_PORT", "29500"))
        cluster = ClusterSpec(tuple(f"{addr}:{port + 23 + k}" for k in range(num_ps)),
                              tuple(f"{addr}:{port + 200 + i}" for i in range(n_workers)))
        if rank < num_ps:
            rdv = Rendezvous(cluster, "ps", rank)
            ps = ParameterServer(cluster, rank, spec, opt, cfg, device=local_rank, rdv=rdv, batch_size=B)
            ps.start()
            # workers register in any order; keep attaching (what `ps.join()` does in the CLI) until all are in
            t_att = time.time()
            while len(ps._attached) < n_workers:
                ps.attach_registered_workers()
                if time.time() - t_att > 240:
                    raise SystemExit(f"ps {rank}: only {len(ps._attached)}/{n_workers} workers registered")
                time.sleep(0.01)
            ps_list = [ps]
        else:
            w = rank - num_ps
            rdv = Rendezvous(cluster, "worker", w)
            worker = Worker(cluster, w, spec, opt, cfg, batch_size=B, device=local_rank, rdv=rdv)
            worker.connect()
            make_loader(worker)
            if worker.is_chief:
                worker.initialize_variables(seed=0)
            worker.wait_ready()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    rdv_any = worker.rdv if worker is not None else ps_list[0].rdv
    phase = [0]
    sync_ms = []

    def full_sync(restart: bool = True, at_rest=None):
        """barrier + torch.cuda.synchronize() on every rank; `at_rest()` runs then, before any serve kernel restarts.

        A resident persistent PS kernel makes a device synchronise hang, and — because CUDA loads kernels lazily —
        even the *first launch* of any new kernel (an NCCL barrier, a torch op) in that context can deadlock
        against it. So: workers quiesce (all their pushes acknowledged) and say so through the TCP store; ps tasks
        then stop their serve kernel (all shard state stays in HBM); only then does every rank run the NCCL
        barrier + synchronise; finally the ps tasks relaunch the kernel and announce it through the store."""
        # (Kept short on purpose: NVLink sublinks drop into a low-power state after tens of milliseconds without
        # traffic and the first pull after that costs ~200 us — measured, profiles/r2/nvlink_idle_probe.log — so the
        # store polls below spin at 0.2 ms instead of sleeping 10 ms.)
        phase[0] += 1
        ph = phase[0]
        t0 = time.perf_counter()
        if worker is not None:
            worker.wait_applied()
        if world > 1:
            if worker is not None:
                rdv_any.add(f"bench/{ph}/quiet", 1)
            if ps_list:
                rdv_any.wait_count(f"bench/{ph}/quiet", n_workers, poll_s=0.0002)
        for ps in ps_list:
            ps.stop()
            if os.environ.get("DM_PS_STATS") == "1":   # serve-kernel counters of the region that just ended (stderr)
                st = ps.serve_stats(reset=True)
                if st:
                    print(f"[ps_stats] sync {ph} rank={rank} shard={ps.task_index} {json.dumps(st)}", file=sys.stderr, flush=True)
        barrier()
        torch.cuda.synchronize()
        if at_rest is not None:
            at_rest()
        if restart:
            for ps in ps_list:
                ps.restart()
            if world > 1:
                if ps_list:
                    rdv_any.add(f"bench/{ph}/serving", 1)
                rdv_any.wait_count(f"bench/{ph}/serving", args.num_ps, poll_s=0.0002)
        sync_ms.append((time.perf_counter() - t0) * 1e3)

    n_rows = xrow = yrow = 0
    if worker is not None:
        assert worker.ld_in == dev_x.shape[1]
        n_rows = dev_x.shape[0] - worker.B_pad
        xrow, yrow = dev_x.shape[1] * dev_x.element_size(), dev_y.shape[1] * 4
    cursor = [0]

    def resident_steps(n, wait_applied=False, timed=False):
        worker.run_resident(n, dev_x.data_ptr(), dev_y.data_ptr(), xrow, yrow, n_rows, cursor[0], wait_applied=wait_applied,
                            **({"timed": True} if timed else {}))
        cursor[0] += n

    def device_timed(n):
        """n steps, CUDA-event timed on the compute stream incl. the ps acknowledgement of the last push (ms)."""
        if engine == "fused":
            # one launch; its tail waits for the acknowledgement of the last push; the two CUDA events are recorded by
            # the native executor on the launching stream immediately before / after the launch
            t_host = time.perf_counter()
            resident_steps(n, wait_applied=True, timed=True)
            enq_ms = (time.perf_counter() - t_host) * 1e3
            return worker.last_elapsed_ms(), enq_ms
        timer = StreamTimer(worker.compute_stream, local_rank)
        timer.start()
        worker.fork_lanes()   # graph engine: no lane starts a timed step before the start event
        t_host = time.perf_counter()
        fused = engine == "fused"
        resident_steps(n, wait_applied=fused)   # fused engine: the launch ends with the acknowledgement wait itself
        enq_ms = (time.perf_counter() - t_host) * 1e3
        if not fused:
            worker.enqueue_wait_ack()
        timer.stop()
        return timer.elapsed_ms(), enq_ms

    def host_fed(n):
        """n steps through Worker.run_steps (gather + H2D + kernels + result read-back), wall clock (s)."""
        t0 = time.perf_counter()
        # returns when every result has been read back and every push of the region is applied on the ps
        outs = worker.run_steps(n, loaders["l"], wait_applied=True)
        dt = time.perf_counter() - t0
        assert len(outs) == n, (len(outs), n)
        return dt

    def dump_outputs():
        """The result of the last device-timed step and the variables the timed steps left on the ps shards (read
        while no serve kernel runs). Larger than DUMP_MAX_BYTES in all: a fixed, seeded sample of every array."""
        if worker is None or not worker.is_chief:
            return
        import numpy as np
        last = worker.last_resident_result()
        arrays = {"loss": np.array([last.loss], np.float32), "correct": np.array([last.correct], np.float32)}
        for name, t in worker.read_variables().items():
            arrays["var_" + name.replace("/", "__")] = t.numpy().astype(np.float32)
        total = sum(a.nbytes for a in arrays.values())
        if total > DUMP_MAX_BYTES:
            rng = np.random.default_rng(0)
            for name, a in arrays.items():
                n = int(a.size * DUMP_MAX_BYTES / total)
                if n < a.size:
                    arrays[name] = a.reshape(-1)[np.sort(rng.choice(a.size, max(n, 1), replace=False))]
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    elapsed_ms = host_enqueue_ms = e2e_s = 0.0
    par = {"dev_ms": 0.0, "e2e_s": 0.0, "strict_ms": 0.0}
    h2d_bytes = d2h_bytes = 0
    launches = 0
    feed_delta = {"direct_chunks": 0, "gathered_chunks": 0, "fills_posted": 0}
    # clocks are sampled from here to the end of the last timed region (started before the warm-up: nvidia-smi's own
    # start-up takes tens of milliseconds and contends for driver locks, which must not sit between the barrier and
    # the first timed launch)
    sampler = ClockSampler(interval_ms=100, gpu_indices=list(range(n_gpus))) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    barrier()
    if worker is not None:
        resident_steps(W)
    full_sync()

    # ---------------- timed region 1: device-timed steps ----------------
    if worker is not None:
        launches_before = worker.kernel_launches()
        elapsed_ms, host_enqueue_ms = device_timed(K)
        launches = worker.kernel_launches() - launches_before + (0 if engine == "fused" else 1)   # (+ wait_ack kernel)
    full_sync(at_rest=dump_outputs if args.dump_outputs else None)
    if os.environ.get("DM_FUSED_DEBUG_TS") == "1" and worker is not None and getattr(worker, "_fx_dbg", None) is not None:
        from bench_tools.fused_phases import print_stamps   # in-kernel phase stamps of the timed launch (stderr)
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):
            print_stamps(worker._fx_dbg.cpu(), f"rank {rank} lanes={args.lanes} K={K}")

    # ---------------- timed region 2: end to end through the public API ----------------
    if not args.skip_e2e:
        if worker is not None:
            worker.run_steps(W, loaders["l"])
        full_sync()
        if worker is not None:
            feed_before = worker.feed_stats()
            e2e_s = host_fed(K)
            feed_after = worker.feed_stats()
            feed_delta = {k: feed_after[k] - feed_before[k] for k in feed_after}
            h2d_bytes = worker.x_bytes + worker.y_bytes
            d2h_bytes = C.sizeof(N.StepResult)
        full_sync()

    # ---------------- reference-semantics lines: one step at a time per worker ----------------
    do_parity = not args.skip_parity and engine == "fused" and args.lanes != 1
    if do_parity:
        if worker is not None:
            worker.set_lanes(1, strict=False)
            resident_steps(W)
            worker.run_steps(W, loaders["l"])
        full_sync()
        if worker is not None:
            par["dev_ms"], _ = device_timed(K)
        full_sync()
        if worker is not None:
            par["e2e_s"] = host_fed(K)
            worker.set_lanes(1, strict=True)
            resident_steps(W)
        full_sync()
        if worker is not None:
            par["strict_ms"], _ = device_timed(K)
            worker.set_lanes(args.lanes, strict=args.strict_steps)
        full_sync()

    if os.environ.get("DM_BENCH_PROBE") == "1" and worker is not None:
        # diagnostic (stderr): cost of the first steps of a launch as a function of the idle time before it
        for gap_ms in (0.0, 0.0, 0.2, 1.0, 5.0, 20.0, 100.0, 0.0):
            if gap_ms:
                time.sleep(gap_ms / 1e3)
            ms20, _ = device_timed(20)
            ms1, _ = device_timed(1)
            print(f"[probe] rank {rank}: idle {gap_ms:6.1f} ms -> 20 steps in {ms20 * 1e3:8.1f} us, then 1 step in "
                  f"{ms1 * 1e3:7.1f} us", file=sys.stderr, flush=True)
    final_step = worker.read_global_step() if (worker is not None and worker.is_chief) else 0
    full_sync(restart=False)   # serve kernels stay down from here on: torch/NCCL ops below are safe
    clocks = sampler.stop() if sampler is not None else None

    # ---------------- reduce over ranks ----------------
    kps = worker.kernels_per_step if worker is not None else 0
    stats = torch.tensor([elapsed_ms, e2e_s, float(launches), float(h2d_bytes), float(d2h_bytes), float(final_step),
                          float(kps), host_enqueue_ms, par["dev_ms"], par["e2e_s"], par["strict_ms"],
                          float(feed_delta["direct_chunks"]), float(feed_delta["gathered_chunks"])],
                         dtype=torch.float64, device="cuda")
    mx = stats.clone()
    sm = stats.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)

    if rank == 0:
        max_ms, max_e2e = float(mx[0]), float(mx[1])
        value = n_workers * K / (max_ms / 1e3)
        n_params = spec.num_params
        peaks = load_peaks()
        # per step: the parameters cross NVLink once in each direction (pull + push), the ps reads the pushed
        # gradient and reads + writes params / m / v (7 x params bytes of HBM/L2 traffic), 2 x fwd + bwd FLOPs
        pbytes = n_params * 4
        flops_step = sum(2 * 2 * B * fi * fo for fi, fo in spec.layer_sizes) + 2 * B * sum(
            fi * fo for fi, fo in spec.layer_sizes[1:])
        per_worker = value / n_workers
        roof = {
            "nvlink_frac": (round(value * pbytes / (NVLINK_GBS * 1e9), 4) if world > 1 else None),
            "nvlink_note": "ps port, each direction: value x param bytes / 770 GB/s (measured peer copy)",
            "hbm_frac": round(value * 7 * pbytes / (peaks["hbm_gbs"] * 1e9), 4),
            "hbm_note": "ps GPU: value x 7 x param bytes (g read, p/m/v read+write) / measured HBM copy bandwidth",
            "tensor_frac": round(per_worker * flops_step / (peaks["bf16_tflops"] * 0.5 * 1e12), 6),
            "tensor_note": "per worker GPU: steps/s x FLOPs/step / (0.5 x measured bf16 peak = tf32 rate)",
            "peaks": peaks,
            "bound": "latency (dependent phases of a 10 MFLOP / 0.64 MB step), not bytes or FLOPs",
        }
        out = {
            "metric": "MNIST-MLP steps/sec (whole box, device-timed, max over ranks)",
            "value": value,
            "unit": "steps/s",
            "n_gpus": n_gpus,
            "steps": K,
            "warmup": W,
            "ms_per_step": max_ms / K,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": ("fp32 storage, tf32 tensor-core multiply, fp32 accumulate" if args.dtype == "fp32" else "bf16"),
            "data": "synthetic",
            "config": {
                "model": f"784-{'-'.join(str(h) for h in spec.hidden)}-10 MLP ({spec.name}), {n_params} params",
                "global_batch": B * n_workers,
                "per_worker_batch": B,
                "seq_len": None,
                "parallelism": (f"{args.num_ps}ps+{n_workers}worker async parameter server"
                                + (" (ps and worker share the GPU)" if world == 1 else " (dedicated ps GPU)")),
                "optimizer": f"{args.optimizer} lr={args.learning_rate}",
                "apply": f"{args.push_mode}/{args.apply_mode}",
                "engine": engine,
                "sharding": args.sharding,
                "steps_in_flight_per_worker": args.lanes,
                "strict_steps": bool(args.strict_steps),
                "mailbox_slots": cfg.nslots,
                "host_enqueue_us_per_step": round(float(mx[7]) * 1e3 / K, 2),
                "l2_policy": "inputs stream from a 55000x784 device-resident dataset (172 MB fp32 > 126 MB L2); "
                             "parameters (0.3 MB) stay L2-resident as in real training",
                "global_step_after_run": int(mx[5]),
                "barrier_sync_ms": [round(v, 2) for v in sync_ms[:3]],
                "host_cores": os.cpu_count(),
                "usable_cores": _usable_cores(),
                "gather_threads_per_worker": os.environ.get("DM_GATHER_THREADS"),
            },
            "clocks": clocks,
            "gpu_launches": int(sm[2]),
            "kernels_per_step": int(mx[6]),
            "steps_per_launch": (K if engine == "fused" else cfg.graph_steps),
            "roofline": roof,
            "impl": "ours",
        }
        if not args.skip_e2e:
            # summed over the workers: how the timed e2e steps got their inputs
            feed_desc = {
                "chunks_from_epoch_buffer": int(sm[11]), "chunks_row_gathered": int(sm[12]),
                "what": "pinned epoch-shuffled dataset buffer -> one contiguous H2D copy per chunk of steps (TF DataSet "
                        "semantics; the next epoch is shuffled into a second pinned buffer by background threads); "
                        "row-gathered chunks go dataset -> pinned staging -> H2D",
            }
            out["e2e"] = {
                "value": n_workers * K / max_e2e,
                "unit": "steps/s",
                "ms_per_step": max_e2e * 1e3 / K,
                "h2d_bytes_per_step": int(mx[3]),
                "d2h_bytes_per_step": int(mx[4]),
                "timing": "wall clock between device synchronisations, max over ranks",
                "input_feed": feed_desc,
            }
        if do_parity:
            out["parity"] = {
                "what": "reference worker semantics: one step at a time per worker (--lanes 1)",
                "value_device_timed": n_workers * K / (float(mx[8]) / 1e3),
                "value_host_fed": n_workers * K / float(mx[9]),
                "value_strict_device_timed": n_workers * K / (float(mx[10]) / 1e3),
                "strict": "--strict_steps: the next pull waits for the ps acknowledgement of the previous push "
                          "(sess.run returns after the apply, reference DS:110-113)",
                "unit": "steps/s",
            }
        print(json.dumps(out), flush=True)

    # ---------------- teardown ----------------
    if inproc is not None:
        inproc.close()
    else:
        if worker is not None:
            worker.finish()
        barrier()
        for ps in ps_list:
            ps.stop()
        if worker is not None:
            worker.close()
        for ps in ps_list:
            ps.close()
        dist.destroy_process_group()
    faulthandler.cancel_dump_traceback_later()
    return 0


if __name__ == "__main__":
    sys.exit(main())
