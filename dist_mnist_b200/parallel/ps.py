"""The parameter-server task.

Reference parity (`/root/reference/distributed_server-basic.py`):
  * DS:80-83   `server = tf.train.Server(...)`; `if job_name == 'ps': server.join()` — a passive process that
               holds the variables, the Adam slots and `global_step` (DS:88-91, 102-103) and executes the
               optimizer apply ops the workers' sessions dispatch to it. It never exits on its own.

Here the shard lives in one GPU's HBM (or in POSIX shm for the CPU backend); a *persistent kernel*
(`ps_serve_kernel`, csrc/ps_apply_sm100.cu) — or the native host loop for the CPU backend — polls the
workers' mailbox flags and applies. The Python object only allocates, publishes the peer-memory descriptor,
attaches workers as they register, and blocks in `join()`.
"""
from __future__ import annotations

import os

import ctypes as C
import threading
import time
from typing import Dict, List, Optional


from .. import _native as N
from ..cluster import ClusterSpec, Rendezvous
from ..models.mlp import MLPSpec
from .config import EngineConfig, OptimizerConfig
from .peer_mem import Carver, Segment
from .sharding import ModelLayout, ShardLayout, build_layout, dw_tile_n_for
from ..utils.metrics import nvtx_annotate

CTRL_GLOBAL_STEP = 0
CTRL_HOST_STOP = 1
CTRL_EXIT_COUNTER = 2
CTRL_WORKER_DONE = 16
CTRL_WORDS = 64


def shard_carver(shard: ShardLayout, n_workers: int, nslots: int) -> Carver:
    """Byte layout of one PS shard segment (both sides derive pointers from the exported table)."""
    a = shard.arena_elems
    ni = max(shard.n_items, 1)
    nf = max(shard.n_flags, 1)
    c = Carver()
    c.add("params", a * 4)
    c.add("adam_m", a * 4)
    c.add("adam_v", a * 4)
    c.add("shadow", a * 2)
    c.add("mailbox", n_workers * nslots * a * 4)
    c.add("flags", n_workers * nslots * nf * 4)
    c.add("next_seq", n_workers * ni * 4)
    c.add("consumed", n_workers * nslots * 4)
    c.add("items", ni * C.sizeof(N.PsItem))
    c.add("item_state", ni * C.sizeof(N.PsItemState))
    c.add("ctrl", CTRL_WORDS * 4)
    c.add("inbox_table", N.MAX_WORKERS * 8)
    c.add("stats", 160 * 8 * 8)      # per-CTA serve statistics (DM_PS_STATS=1)
    return c


class ParameterServer:
    def __init__(self, cluster: ClusterSpec, task_index: int, spec: MLPSpec, opt: OptimizerConfig,
                 cfg: EngineConfig, device: int = 0, rdv: Optional[Rendezvous] = None,
                 layout: Optional[ModelLayout] = None, verbose: bool = False, batch_size: int = 32):
        cfg.validate(opt)
        if cluster.num_workers > N.MAX_WORKERS:
            raise ValueError(f"at most {N.MAX_WORKERS} workers per ps shard")
        self.cluster, self.task_index, self.spec, self.opt, self.cfg = cluster, task_index, spec, opt, cfg
        self.device = device if cfg.backend == "cuda" else -1
        self.verbose = verbose
        # the shard tiling follows the step engine the workers will use (same rule, same flags on both sides)
        self.engine = layout.engine if layout is not None else cfg.resolve_engine(spec, batch_size)
        self.layout = layout or build_layout(spec, cluster.num_ps, cfg.sharding, dw_tile_n_for(cfg.dtype),
                                             engine=self.engine, ps_row_blocks=cfg.ps_row_blocks)
        self.shard = self.layout.shards[task_index]
        self.rdv = rdv or Rendezvous(cluster, "ps", task_index)
        self.n_workers = cluster.num_workers
        self.lib = N.lib()
        self._attached: Dict[int, Segment] = {}
        self._attached_device: Dict[int, int] = {}   # worker -> CUDA device of its current incarnation
        self._serving = False
        self._cpu_handle = None
        self._stream = None
        self._ctl_stream = None
        self._pin = None
        self._cpu_table = (C.c_void_p * N.MAX_WORKERS)() if cfg.backend == "cpu" else None
        self._lock = threading.Lock()
        self._dead = set()          # workers declared dead by the failure detector
        self._attached_at: Dict[int, float] = {}   # worker -> time its current incarnation was attached
        self._incarnation: Dict[int, int] = {}   # worker -> incarnation number currently attached
        self._readmit_restart = False

        kind = "cuda" if cfg.backend == "cuda" else "shm"
        if kind == "cuda":
            N.check(self.lib.dm_set_device(self.device), "set device")
        carver = shard_carver(self.shard, self.n_workers, cfg.nslots)
        self.seg = Segment.create(kind, carver.total, device=self.device, table=carver.table(), tag=f"ps{task_index}")
        self._init_tables()
        desc = self.seg.export()
        desc.update({
            "arena_elems": self.shard.arena_elems, "n_items": self.shard.n_items, "n_flags": self.shard.n_flags,
            "nslots": cfg.nslots, "engine": self.engine,
            "n_workers": self.n_workers, "owns_global_step": self.shard.owns_global_step,
        })
        self.rdv.put(f"ps/{task_index}/segment", desc)

    # ------------------------------------------------------------------------------------------
    def _host_write(self, region: str, data: bytes, byte_offset: int = 0) -> None:
        """Synchronous host -> segment write (setup time only)."""
        if self.cfg.backend == "cuda":
            buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
            N.check(self.lib.dm_memcpy_async(self.seg.addr(region, byte_offset), C.addressof(buf), len(data), None))
            N.check(self.lib.dm_stream_sync(None))
        else:
            C.memmove(self.seg.addr(region, byte_offset), data, len(data))

    def _init_tables(self) -> None:
        sh = self.shard
        ni = max(sh.n_items, 1)
        items = (N.PsItem * ni)()
        for i, it in enumerate(sh.items):
            items[i].offset, items[i].rows, items[i].cols, items[i].ld = it.offset, it.rows, it.cols, it.ld
            items[i].flags = 1 if (it.shadow and self.cfg.dtype == "bf16") else 0
            items[i].flag_index = it.flag if it.flag >= 0 else i
        self._host_write("items", bytes(items))
        self.reset_optimizer_state()
        ones = (C.c_uint32 * (self.n_workers * ni))(*([1] * (self.n_workers * ni)))
        self._host_write("next_seq", bytes(ones))

    def reset_optimizer_state(self) -> None:
        ni = max(self.shard.n_items, 1)
        st = (N.PsItemState * ni)()
        for i in range(ni):
            st[i].t, st[i].beta1_pow, st[i].beta2_pow = 0, 1.0, 1.0
        self._host_write("item_state", bytes(st))

    # ------------------------------------------------------------------------------------------
    def _serve_params(self) -> N.PsServeParams:
        s, sh, cfg, opt = self.seg, self.shard, self.cfg, self.opt
        P = N.PsServeParams()
        P.params, P.adam_m, P.adam_v = s.addr("params"), s.addr("adam_m"), s.addr("adam_v")
        P.shadow_bf16 = s.addr("shadow") if cfg.dtype == "bf16" else None
        P.items, P.item_state = s.addr("items"), s.addr("item_state")
        P.n_items, P.n_workers, P.nslots = sh.n_items, self.n_workers, cfg.nslots
        P.n_flags = max(sh.n_flags, 1)
        P.oneshot = 0
        P.opt, P.apply_mode = opt.native_kind, cfg.native_apply_mode
        P.lr, P.beta1, P.beta2, P.eps = opt.lr, opt.beta1, opt.beta2, opt.eps
        P.ieee_math = 1 if opt.math == "ieee" else 0
        P.mailbox, P.arena_elems = s.addr("mailbox"), sh.arena_elems
        P.flags, P.next_seq, P.consumed = s.addr("flags"), s.addr("next_seq"), s.addr("consumed")
        P.global_step = s.addr("ctrl", 4 * CTRL_GLOBAL_STEP)
        P.host_stop = s.addr("ctrl", 4 * CTRL_HOST_STOP)
        P.exit_counter = s.addr("ctrl", 4 * CTRL_EXIT_COUNTER)
        P.worker_done = s.addr("ctrl", 4 * CTRL_WORKER_DONE)
        # flags / acks need system scope only when some worker sits on another GPU
        P.lookahead = int(os.environ.get("DM_PS_LOOKAHEAD", "0"))
        P.stats = s.addr("stats") if (cfg.backend == "cuda" and os.environ.get("DM_PS_STATS") == "1") else None
        devs = list(self._attached_device.values())
        P.gpu_scope = int(cfg.backend == "cuda" and self.n_workers == 1 and len(devs) == 1 and devs[0] == self.device)
        if cfg.backend == "cuda":
            P.inbox_table = s.addr("inbox_table")
        else:
            P.inbox_table = C.addressof(self._cpu_table)
        return P

    @nvtx_annotate("dm.ps.start")
    def start(self, wait_init: bool = True, timeout_s: Optional[float] = None) -> None:
        """Begin serving. Waits (like TF's non-chief `ready_op` poll) until the chief has initialised the
        variables, then launches the serve kernel / loop and announces `ps/<k>/serving`."""
        if self._serving:
            return
        if wait_init:
            self.rdv.get("init/done", timeout_s)
        self.attach_registered_workers()
        if self.cfg.push_mode == "atomic":
            # async-SGD red.add mode: the worker kernels apply straight into the master copy; the shard is pure
            # memory + the L2 atomic units, no serve kernel is needed.
            self._serving = True
            self.rdv.put(f"ps/{self.task_index}/serving", {"mode": "atomic"})
            return
        P = self._serve_params()
        self._P = P
        self.oneshot = self.cfg.ps_mode == "oneshot" and self.cfg.backend == "cuda"
        if self.cfg.backend == "cuda":
            N.check(self.lib.dm_set_device(self.device), "set device")
            N.ensure_prepared(self.device)  # load every kernel before the persistent one becomes resident
            out = C.c_void_p()
            N.check(self.lib.dm_stream_create(C.byref(out)))
            self._stream = out.value
            N.check(self.lib.dm_stream_create(C.byref(out)))
            self._ctl_stream = out.value
            N.check(self.lib.dm_host_alloc(4096, C.byref(out)))
            self._pin = out.value
            if self.oneshot:
                P.oneshot = 1   # nothing resident: `serve_once()` runs the kernel after the workers' kernels
            else:
                n_ctas = self._serve_ctas()
                N.check(self.lib.dm_launch_ps_serve(C.addressof(P), n_ctas, self._stream), "launch ps_serve")
        else:
            self._cpu_handle = self.lib.dm_cpu_ps_start(C.addressof(P))
        self._serving = True
        self.rdv.put(f"ps/{self.task_index}/serving", {"mode": "oneshot" if self.oneshot else "mailbox"})

    @nvtx_annotate("dm.ps.serve_once")
    def serve_once(self, after_stream: Optional[int] = None, wait: bool = True) -> None:
        """One-shot mode: launch the serve kernel once; it applies every push that is complete in memory and exits
        after the first sweep that finds nothing (csrc/ps_apply_sm100.cu, PsServeParams::oneshot). `after_stream`:
        a CUDA stream whose enqueued work (the worker's step kernels) must finish first — the launch is ordered
        behind it with an event, so nothing ever waits for a kernel that has not been launched: safe under
        profilers and sanitizers that serialise kernels."""
        if not getattr(self, "oneshot", False) or not self._serving:
            return
        if after_stream is not None:
            N.check(self.lib.dm_stream_wait_stream(self._stream, after_stream), "order serve after worker")
        N.check(self.lib.dm_launch_ps_serve(C.addressof(self._P), self._serve_ctas(), self._stream), "launch ps_serve")
        if wait:
            N.check(self.lib.dm_stream_sync(self._stream), "one-shot ps serve kernel")

    # ------------------------------------------------------------------------------------------
    def _patch_table(self, w: int, ptr: int) -> None:
        if self.cfg.push_mode == "atomic":
            return
        if self.cfg.backend == "cuda":
            if self._serving:
                # the serve kernel is running: patch through the side stream from pinned memory
                C.c_uint64.from_address(self._pin + 8 * w).value = ptr
                N.check(self.lib.dm_memcpy_async(self.seg.addr("inbox_table", 8 * w), self._pin + 8 * w, 8,
                                                 self._ctl_stream))
                N.check(self.lib.dm_stream_sync(self._ctl_stream))
            else:
                self._host_write("inbox_table", bytes(C.c_uint64(ptr)), 8 * w)
        else:
            self._cpu_table[w] = ptr

    def attach_registered_workers(self) -> List[int]:
        """Map the inbox of every worker that has registered since the last call (late joiners welcome)."""
        new = []
        with self._lock:
            for w in range(self.n_workers):
                if w in self._attached and self.rdv.add(f"worker/{w}/incarnation", 0) == self._incarnation.get(w):
                    continue
                desc = self.rdv.try_get(f"worker/{w}/inbox")
                if desc is None or desc.get("incarnation", 1) == self._incarnation.get(w):
                    continue
                if w in self._attached:
                    self._readmit(w)       # a restarted worker: forget everything about its previous life
                seg = Segment.open(desc, device=self.device)
                self._attached[w] = seg
                self._incarnation[w] = desc.get("incarnation", 1)
                self._attached_device[w] = desc.get("worker_device", -1)
                self._attached_at[w] = time.time()
                ptr = seg.addr("inbox", 8 * desc["inbox_index"][str(self.task_index)]) \
                    if str(self.task_index) in desc["inbox_index"] else 0
                if ptr:
                    self._patch_table(w, ptr)
                if self._readmit_restart:
                    self._readmit_restart = False
                    self.restart()
                self.rdv.put(f"ps/{self.task_index}/attached/{w}/{self._incarnation[w]}", True)
                new.append(w)
        return new

    @nvtx_annotate("dm.ps.readmit")
    def _readmit(self, w: int) -> None:
        """Elastic recovery: worker `w` crashed and was started again. Its new life begins with push sequence 1 and
        a new inbox, so this shard drops the old incarnation's bookkeeping: the serve kernel is stopped (its
        per-worker cursors live in shared memory), flags / consumed counters / cursors / the done word of `w` are
        reset, and serving resumes. Parameters, optimizer state and global_step are untouched."""
        print(f"[ps {self.task_index}] worker {w} re-registered (incarnation "
              f"{self.rdv.add(f'worker/{w}/incarnation', 0)}): re-admitting it", flush=True)
        old = self._attached.pop(w)
        self._attached_device.pop(w, None)
        if self.cfg.push_mode == "atomic":
            try:
                old.close()
            except Exception:
                pass               # the process that exported it is gone
            if w in self._dead and self.task_index == 0:
                self.rdv.add("session/workers_done", -1)
            self._dead.discard(w)
            return
        # order matters: the serve loop / kernel may still acknowledge an old push into the previous incarnation's
        # inbox, so it is stopped and the table entry cleared *before* that mapping goes away
        was_serving = self._serving and not getattr(self, "oneshot", False)
        if was_serving:
            self.stop()
        self._patch_table(w, 0)
        try:
            old.close()
        except Exception:
            pass                   # the process that exported it is gone
        ni, ns, nf = max(self.shard.n_items, 1), self.cfg.nslots, max(self.shard.n_flags, 1)
        self._host_write("flags", bytes(4 * ns * nf), 4 * w * ns * nf)
        self._host_write("consumed", bytes(4 * ns), 4 * w * ns)
        self._host_write("next_seq", bytes((C.c_uint32 * ni)(*([1] * ni))), 4 * w * ni)
        self._host_write("ctrl", bytes(4), 4 * (CTRL_WORKER_DONE + w))
        self._dead.discard(w)
        self._readmit_restart = was_serving

    # ------------------------------------------------------------------------------------------
    def kernel_running(self) -> bool:
        if not self._serving or self.cfg.push_mode == "atomic" or getattr(self, "oneshot", False):
            return False
        if self.cfg.backend == "cuda":
            return self.lib.dm_stream_query(self._stream) == 1
        return self._cpu_handle is not None and self.lib.dm_cpu_ps_running(self._cpu_handle) == 1

    def global_step(self) -> int:
        if self.cfg.backend == "cuda":
            host = C.c_uint32(0)
            stream = self._ctl_stream
            N.check(self.lib.dm_memcpy_async(C.addressof(host), self.seg.addr("ctrl", 4 * CTRL_GLOBAL_STEP), 4, stream))
            N.check(self.lib.dm_stream_sync(stream))
            return host.value
        return self.lib.dm_load_acquire_u32(self.seg.addr("ctrl", 4 * CTRL_GLOBAL_STEP))

    @nvtx_annotate("dm.ps.stop")
    def stop(self) -> None:
        """Ask the serve kernel / loop to exit and wait for it."""
        if not self._serving:
            return
        if self.cfg.push_mode != "atomic" and getattr(self, "oneshot", False):
            N.check(self.lib.dm_stream_sync(self._stream), "one-shot ps serve kernel")
        elif self.cfg.push_mode != "atomic":
            if self.cfg.backend == "cuda":
                C.c_uint32.from_address(self._pin + 1024).value = 1
                N.check(self.lib.dm_memcpy_async(self.seg.addr("ctrl", 4 * CTRL_HOST_STOP), self._pin + 1024, 4,
                                                 self._ctl_stream))
                N.check(self.lib.dm_stream_sync(self._ctl_stream))
                N.check(self.lib.dm_stream_sync(self._stream), "ps serve kernel")
            else:
                self.lib.dm_store_release_u32(self.seg.addr("ctrl", 4 * CTRL_HOST_STOP), 1)
                self.lib.dm_cpu_ps_join(self._cpu_handle)
                self._cpu_handle = None
        self._serving = False

    def serve_stats(self, reset: bool = False) -> Optional[dict]:
        """Aggregated serve-kernel statistics (DM_PS_STATS=1; valid after stop()): per-pass averages over CTAs.
        `reset`: zero the counters afterwards (per-region statistics)."""
        if self.cfg.backend != "cuda" or os.environ.get("DM_PS_STATS") != "1":
            return None
        n = 160 * 8
        host = (C.c_uint64 * n)()
        N.check(self.lib.dm_memcpy_async(C.addressof(host), self.seg.addr("stats"), 8 * n, None))
        N.check(self.lib.dm_stream_sync(None))
        if reset:
            zeros = (C.c_uint64 * n)()
            N.check(self.lib.dm_memcpy_async(self.seg.addr("stats"), C.addressof(zeros), 8 * n, None))
            N.check(self.lib.dm_stream_sync(None))
        rows = [list(host[i * 8:(i + 1) * 8]) for i in range(160) if host[i * 8] or host[i * 8 + 4]]
        if not rows:
            return None
        tot = [sum(r[j] for r in rows) for j in range(8)]
        khz = C.c_int(0)
        N.check(self.lib.dm_device_clock_khz(self.device, C.byref(khz)))
        mhz = khz.value / 1e3   # the device's maximum SM clock: cycle counts -> lower-bound microseconds
        return {
            "ctas": len(rows), "passes": tot[0], "pushes": tot[1],
            "pushes_per_pass": round(tot[1] / max(tot[0], 1), 2), "max_pushes_in_pass": max(r[6] for r in rows),
            "apply_us_per_pass": round(tot[2] / max(tot[0], 1) / mhz, 2),
            "bookkeeping_us_per_pass": round(tot[3] / max(tot[0], 1) / mhz, 2),
            "poll_us_per_working_pass": round(tot[7] / max(tot[0], 1) / mhz, 2),
            "idle_polls": tot[4], "idle_poll_us": round(tot[5] / max(tot[4], 1) / mhz, 2),
            "busy_fraction": round((tot[2] + tot[3] + tot[7]) / max(tot[2] + tot[3] + tot[7] + tot[5], 1), 3),
        }

    def _serve_ctas(self) -> int:
        """One item per CTA where possible: a dedicated ps GPU gives the serve kernel (almost) every SM, a GPU
        shared with a worker keeps most SMs for the worker's step kernels."""
        want = self.cfg.ps_ctas
        if want <= 0:
            shared = any(d == self.device for d in self._attached_device.values())
            want = 40 if shared else 128
        return max(1, min(want, self.shard.n_items))

    def restart(self) -> None:
        """Relaunch the serve kernel / loop after `stop()` (all shard state lives in the segment, so serving
        resumes exactly where it stopped). Used by the benchmark to bracket timed regions with a full device
        synchronise, which a running persistent kernel would never let return."""
        if self._serving:
            return
        if self.cfg.push_mode == "atomic":
            self._serving = True
            return
        if getattr(self, "oneshot", False):
            self._serving = True
            return
        if self.cfg.backend == "cuda":
            N.check(self.lib.dm_set_device(self.device), "set device")
            N.check(self.lib.dm_memset_async(self.seg.addr("ctrl", 4 * CTRL_HOST_STOP), 0, 4, self._ctl_stream))
            N.check(self.lib.dm_stream_sync(self._ctl_stream))
            n_ctas = self._serve_ctas()
            N.check(self.lib.dm_launch_ps_serve(C.addressof(self._P), n_ctas, self._stream), "launch ps_serve")
        else:
            self.lib.dm_store_release_u32(self.seg.addr("ctrl", 4 * CTRL_HOST_STOP), 0)
            self._cpu_handle = self.lib.dm_cpu_ps_start(C.addressof(self._P))
        self._serving = True

    def _worker_done_word(self, w: int) -> int:
        addr = self.seg.addr("ctrl", 4 * (CTRL_WORKER_DONE + w))
        if self.cfg.backend == "cuda":
            host = C.c_uint32(0)
            N.check(self.lib.dm_memcpy_async(C.addressof(host), addr, 4, self._ctl_stream))
            N.check(self.lib.dm_stream_sync(self._ctl_stream))
            return host.value
        return self.lib.dm_load_acquire_u32(addr)

    def mark_worker_dead(self, w: int) -> None:
        """Failure handling: stop waiting for worker `w` (its half-finished push, if any, is dropped; everything it
        pushed completely stays applied). Asynchronous training means the other workers never depended on it."""
        self._patch_table(w, 0)     # no more acknowledgements into the dead process's memory
        addr = self.seg.addr("ctrl", 4 * (CTRL_WORKER_DONE + w))
        if self.cfg.backend == "cuda":
            C.c_uint32.from_address(self._pin + 1028).value = N.WORKER_DEAD
            N.check(self.lib.dm_memcpy_async(addr, self._pin + 1028, 4, self._ctl_stream))
            N.check(self.lib.dm_stream_sync(self._ctl_stream))
        else:
            self.lib.dm_store_release_u32(addr, N.WORKER_DEAD)
        self._dead.add(w)

    def revive_worker(self, w: int) -> None:
        """Undo `mark_worker_dead` for a worker whose heartbeat resumed (it was slow, not dead): its inbox pointer is
        restored and the serve loop waits for its pushes again. Pushes it completed meanwhile were applied anyway —
        only the acknowledgements were suppressed."""
        seg = self._attached.get(w)
        if seg is None:
            return
        desc = self.rdv.try_get(f"worker/{w}/inbox") or {}
        idx = desc.get("inbox_index", {}).get(str(self.task_index))
        addr = self.seg.addr("ctrl", 4 * (CTRL_WORKER_DONE + w))
        if self.cfg.backend == "cuda":
            C.c_uint32.from_address(self._pin + 1032).value = 0
            N.check(self.lib.dm_memcpy_async(addr, self._pin + 1032, 4, self._ctl_stream))
            N.check(self.lib.dm_stream_sync(self._ctl_stream))
        else:
            self.lib.dm_store_release_u32(addr, 0)
        if idx is not None:
            self._patch_table(w, seg.addr("inbox", 8 * idx))
        self._dead.discard(w)
        print(f"[ps {self.task_index}] worker {w} is alive again (heartbeat resumed)", flush=True)

    def check_worker_liveness(self, timeout_s: float) -> List[int]:
        """Declare dead every attached worker that has neither finished nor sent a heartbeat for `timeout_s`
        seconds (workers heartbeat through the rendezvous store once per train-loop chunk). Returns the workers
        newly declared dead."""
        newly = []
        now = time.time()
        for w in list(self._attached):
            hb = self.rdv.try_get(f"session/heartbeat/{w}")
            if w in self._dead:
                # a worker that was only slow (long graph capture, a paused process) heartbeats again: take it back
                if hb is not None and now - float(hb) <= timeout_s and self.cfg.push_mode != "atomic":
                    self.revive_worker(w)
                continue
            # the liveness clock starts when this incarnation was attached by *this* shard, not at its first heartbeat
            # (a non-chief worker connects long before the chief has finished initialising)
            last = max(float(hb) if hb is not None else 0.0, self._attached_at.get(w, now))
            if hb is None or now - last <= timeout_s:
                continue
            if self.cfg.push_mode != "atomic" and self._worker_done_word(w) != 0:
                continue   # it left the session cleanly
            if self.cfg.push_mode == "atomic" and self.rdv.try_get(f"session/done/{w}") is not None:
                continue
            print(f"[ps {self.task_index}] worker {w} presumed dead: no heartbeat for {now - float(hb):.1f} s; "
                  f"serving the remaining workers", flush=True)
            if self.cfg.push_mode != "atomic":
                self.mark_worker_dead(w)
            else:
                self._dead.add(w)
                if self.task_index == 0:
                    self.rdv.add("session/workers_done", 1)
            newly.append(w)
        return newly

    def join(self, exit_when_done: bool = False, poll_s: float = 0.05, worker_timeout_s: float = 0.0) -> None:
        """`server.join()` (DS:83): block forever serving. With `exit_when_done` the call returns once every
        worker has left the session (or is presumed dead, `worker_timeout_s > 0`) and all their pushes are applied,
        or when a `shutdown` mark appears."""
        last_check = time.time()
        while True:
            self.attach_registered_workers()
            if self.rdv.try_get("shutdown") is not None:
                break
            if worker_timeout_s > 0 and time.time() - last_check >= min(1.0, worker_timeout_s / 2):
                last_check = time.time()
                self.check_worker_liveness(worker_timeout_s)
            if exit_when_done:
                if self.cfg.push_mode == "atomic":
                    if self.rdv.add("session/workers_done", 0) >= self.n_workers:
                        break
                elif getattr(self, "oneshot", False):
                    if self.rdv.add("session/workers_done", 0) >= self.n_workers:
                        self.serve_once()
                        break
                elif self._serving and not self.kernel_running():
                    break
            if getattr(self, "oneshot", False):
                self.serve_once()      # one-shot mode as a stand-alone task: apply whatever has arrived
            time.sleep(poll_s)
        self.stop()
        if exit_when_done:
            self._leave_rendezvous()

    def _leave_rendezvous(self, timeout_s: float = 30.0) -> None:
        """ps 0 hosts the rendezvous store, so it keeps it up until the other tasks have made their last call to it:
        the other ps tasks leave their serve loops at about the same time and poll the store until then, and a worker
        adds to `session/workers_done` only after its done word has reached the shards. Bounded: a task that died
        never signs off."""
        if not self.rdv.is_master:
            self.rdv.add("session/ps_left", 1)
            return
        deadline = time.time() + timeout_s
        while (self.rdv.add("session/ps_left", 0) < self.cluster.num_ps - 1
               or self.rdv.add("session/workers_done", 0) + len(self._dead) < self.n_workers):
            if time.time() > deadline:
                break
            time.sleep(0.01)

    def close(self) -> None:
        self.stop()
        for seg in self._attached.values():
            seg.close()
        self._attached.clear()
        if self.cfg.backend == "cuda":
            if self._stream:
                self.lib.dm_stream_destroy(self._stream)
                self.lib.dm_stream_destroy(self._ctl_stream)
                self.lib.dm_host_free(self._pin)
                self._stream = self._ctl_stream = self._pin = None
        self.seg.close()
