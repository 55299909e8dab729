"""The worker task: between-graph replicated, asynchronous data-parallel training against the PS shards.

Reference parity (`/root/reference/distributed_server-basic.py`):
  * DS:87-103   each worker builds its *own* replica of the model; variables live on the ps tasks.
  * DS:108-109  `MonitoredTrainingSession(master, is_chief=(task_index == 0), ...)`: worker 0 initialises the
                variables (or restores a checkpoint), the others wait until that has happened.
  * DS:110-113  one step = pull variables, forward/backward on the worker, push gradients, PS applies Adam and
                bumps `global_step`; the worker gets `loss` and `global_step` back. No locks, no barriers.

GPU backend, two step engines (`EngineConfig.engine`, resolved by `EngineConfig.resolve_engine`):
  * "fused" (784-H-10 models, H <= 128, batch <= 32, fp32 — the reference's live configuration): whole steps run
    inside one persistent kernel (csrc/fused_step_sm100.cu): an 8-CTA cluster pulls its K-slices of W from the ps
    shard(s) with TMA over NVLink, tcgen05 forward with a DSMEM reduce-scatter, head, DSMEM all-gather, tcgen05 dW
    whose epilogue pushes into the ps mailbox; `cfg.lanes` clusters work on different steps concurrently. The
    native executor (csrc/fused_exec.cu) feeds it chunk by chunk: gather pool -> pinned staging -> H2D -> one launch.
  * "graph" (any depth / width / bf16): a PDL-linked chain of per-layer kernels inside a CUDA graph (`ops/`,
    csrc/gemm_sm100.cu, csrc/head_sm100.cu) driven by csrc/executor.cu.

CPU backend: same protocol over POSIX shm with torch CPU math (BASELINE.json config 1, plumbing tests).
"""
from __future__ import annotations

import collections.abc
import ctypes as C
import os
import time
import weakref
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import _native as N
from ..cluster import ClusterSpec, Rendezvous
from ..models import mlp
from ..models.mlp import MLPSpec
from ..ops import gemm as gemm_ops
from ..ops import head as head_ops
from .config import MAX_SLOTS, EngineConfig, OptimizerConfig
from .peer_mem import Carver, Segment
from .ps import CTRL_GLOBAL_STEP, CTRL_WORKER_DONE
from .sharding import FUSED_CLUSTER, ModelLayout, VarLayout, build_layout, dw_tile_n_for
from ..utils.metrics import nvtx_annotate


@dataclass
class StepOutput:
    loss: float
    global_step: int
    correct: int
    seq: int


_STEP_DTYPE = np.dtype([("loss", np.float32), ("global_step", np.uint32), ("correct", np.uint32), ("seq", np.uint32)])


class StepOutputs(collections.abc.Sequence):
    """Results of a native run of steps: a read-only sequence of `StepOutput` backed by the executor's result
    array (no per-step Python object is built unless the step is looked at). `.loss`, `.global_step`, `.correct`
    and `.seq` give the whole columns as numpy arrays."""

    def __init__(self, raw: np.ndarray):
        self._raw = raw

    def __len__(self) -> int:
        return int(self._raw.shape[0])

    def __getitem__(self, i):
        if isinstance(i, slice):
            return StepOutputs(self._raw[i])
        r = self._raw[i]
        return StepOutput(float(r["loss"]), int(r["global_step"]), int(r["correct"]), int(r["seq"]))

    loss = property(lambda self: self._raw["loss"])
    global_step = property(lambda self: self._raw["global_step"])
    correct = property(lambda self: self._raw["correct"])
    seq = property(lambda self: self._raw["seq"])


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def usable_cores() -> int:
    """CPU cores this process may really use: the affinity mask, further limited by a cgroup CPU quota (a container
    can see 128 cores and be throttled to a fraction of them — spinning helper threads beyond the quota stall the
    whole process for the rest of every scheduler period)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 8
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // period))
            break
        except Exception:
            continue
    return n


class Worker:
    def __init__(self, cluster: ClusterSpec, task_index: int, spec: MLPSpec, opt: OptimizerConfig,
                 cfg: EngineConfig, batch_size: int = 32, device: int = 0, rdv: Optional[Rendezvous] = None,
                 layout: Optional[ModelLayout] = None, verbose: bool = False):
        cfg.validate(opt)
        if batch_size < 1 or batch_size > 256:
            raise ValueError("batch_size must be in [1, 256] per worker")
        if spec.num_classes > head_ops.MAX_CLASSES:
            raise ValueError(f"at most {head_ops.MAX_CLASSES} classes")
        self.cluster, self.task_index, self.spec, self.opt, self.cfg = cluster, task_index, spec, opt, cfg
        self.batch = batch_size
        self.B_pad = _round_up(batch_size, 16)
        self.device = device if cfg.backend == "cuda" else -1
        self.verbose = verbose
        self.engine = layout.engine if layout is not None else cfg.resolve_engine(spec, batch_size)
        self.layout = layout or build_layout(spec, cluster.num_ps, cfg.sharding, dw_tile_n_for(cfg.dtype),
                                             engine=self.engine, ps_row_blocks=cfg.ps_row_blocks)
        if self.engine == "fused":
            self.B_pad = N.FUSED_ROWS_PER_SLOT   # the fused kernel always works on 32-row tiles (rows >= batch masked)
        self.rdv = rdv or Rendezvous(cluster, "worker", task_index)
        self.lib = N.lib()
        self.is_chief = task_index == 0  # DS:108
        self.ps_segs: List[Segment] = []
        self.seg: Optional[Segment] = None
        self._exec = None
        self._fexec = None          # fused engine: native executor handle (csrc/fused_exec.cu)
        self._ps_local: List = []   # in-process clusters with one-shot ps tasks: serve after every launch
        self._connected = False
        self._closed = False
        self._seq_host = 0          # cpu backend: push sequence number
        self.dt = cfg.native_dtype
        self.es = gemm_ops.elem_size(self.dt)
        self.tdtype = torch.float32 if cfg.dtype == "fp32" else torch.bfloat16
        self.ld_in = gemm_ops.padded_ld(spec.in_features)
        # shards this worker pushes to, the one owning global_step first (its inbox entry is index 0)
        used = [sh.ps for sh in self.layout.shards if sh.n_items > 0]
        gs_owner = self.layout.placement["global_step"]
        # The shared step counter is the one of the first shard in `inbox_order` (its serve loop counts fully applied
        # pushes and reports the count with every acknowledgement). Normally that is the shard placement gives
        # `global_step` to; when that shard owns no variable at all (more ps tasks than variables) no serve loop ever
        # increments its counter, so the counter of the first shard that does own items is authoritative instead.
        self.gs_owner = gs_owner if (gs_owner in used or not used) else used[0]
        gs_owner = self.gs_owner
        self.inbox_order = ([gs_owner] if gs_owner in used else []) + [k for k in used if k != gs_owner]
        self.inbox_index = {k: i for i, k in enumerate(self.inbox_order)}
        self.kernels_per_step = 0

    # ------------------------------------------------------------------------------------------
    # bring-up
    # ------------------------------------------------------------------------------------------
    def connect(self, timeout_s: Optional[float] = None) -> None:
        """Open every PS shard, publish our inbox, and (non-chief) wait for the chief's initialisation."""
        cfg = self.cfg
        if cfg.backend == "cuda":
            N.check(self.lib.dm_set_device(self.device), "set device")
            torch.cuda.set_device(self.device)
        self.ps_desc = []
        for k in range(self.cluster.num_ps):
            desc = self.rdv.get(f"ps/{k}/segment", timeout_s)
            if desc["nslots"] != cfg.nslots or desc["n_workers"] != self.cluster.num_workers:
                raise RuntimeError(f"ps {k} was started with a different engine configuration: {desc}")
            sh = self.layout.shards[k]
            if (desc["arena_elems"] != sh.arena_elems or desc["n_items"] != sh.n_items
                    or desc.get("n_flags", sh.n_flags) != sh.n_flags or desc.get("engine", self.engine) != self.engine):
                raise RuntimeError(f"ps {k} has a different model layout (model / batch_size / sharding / engine "
                                   f"flags differ?): ps {desc.get('engine')} {desc['n_items']} items, "
                                   f"worker {self.engine} {sh.n_items} items")
            self.ps_desc.append(desc)
            self.ps_segs.append(Segment.open(desc, device=self.device))
        carver = Carver()
        carver.add("inbox", max(1, len(self.inbox_order)) * 8)
        carver.add("seq", 4 * (1 + MAX_SLOTS))   # [0] pushes opened so far, [1 + slot] seq of the slot's current step
        kind = "cuda" if cfg.backend == "cuda" else "shm"
        self.seg = Segment.create(kind, carver.total, device=self.device, table=carver.table(),
                                  tag=f"w{self.task_index}")
        desc = self.seg.export()
        desc["inbox_index"] = {str(k): i for k, i in self.inbox_index.items()}
        desc["worker_device"] = self.device
        # a worker that is restarted after a crash registers again under the next incarnation number; the ps
        # tasks then re-admit it (fresh push sequence, fresh inbox) — the reference's recoverable session
        self.incarnation = self.rdv.add(f"worker/{self.task_index}/incarnation", 1)
        desc["incarnation"] = self.incarnation
        self.rdv.put(f"worker/{self.task_index}/inbox", desc)
        self.heartbeat()
        self._start_heartbeat_thread()
        self._connected = True

    @nvtx_annotate("dm.worker.wait_ready")
    def wait_ready(self, timeout_s: Optional[float] = None) -> None:
        """Block until the variables are initialised (DS:108-109 non-chief wait) and every PS shard serves us."""
        self.rdv.get("init/done", timeout_s)
        for k in range(self.cluster.num_ps):
            self.rdv.get(f"ps/{k}/serving", timeout_s)
            self.rdv.get(f"ps/{k}/attached/{self.task_index}/{self.incarnation}", timeout_s)
        self.heartbeat()
        self.prepare()
        self.heartbeat()
        # seed our view of the shared step counter (a restored session does not start at 0)
        g0 = self.read_global_step()
        if self.cfg.backend == "cuda":
            host = C.c_uint32(g0)
            N.check(self.lib.dm_memcpy_async(self.seg.addr("inbox", 4), C.addressof(host), 4, None))
            N.check(self.lib.dm_stream_sync(None))
        else:
            self.lib.dm_store_release_u32(self.seg.addr("inbox", 4), g0)

    def _read_own(self, region: str, count: int, byte_offset: int = 0) -> List[int]:
        if self.cfg.backend == "cuda":
            host = (C.c_uint32 * count)()
            N.check(self.lib.dm_memcpy_async(C.addressof(host), self.seg.addr(region, byte_offset), 4 * count, None))
            N.check(self.lib.dm_stream_sync(None))
            return list(host)
        return [self.lib.dm_load_acquire_u32(self.seg.addr(region, byte_offset + 4 * i)) for i in range(count)]

    def _seq_word_ptr(self) -> int:
        """Device word holding the number of pushes this worker has made (read by wait_ack / worker_done kernels)."""
        if self.engine == "fused" and self._fexec:
            return self._fx_ctl + 8
        return self.seg.addr("seq")

    def pushes_made(self) -> int:
        if self.cfg.backend == "cuda":
            self.drain()
            if self.engine == "fused":
                return int(self.lib.dm_fexec_steps_done(self._fexec)) if self._fexec else 0
            return self._read_own("seq", 1)[0]
        return self._seq_host

    @nvtx_annotate("dm.worker.wait_applied")
    def wait_applied(self, timeout_s: float = 60.0) -> None:
        """Block until every push this worker has made is applied on every shard (needed for a consistent
        checkpoint or evaluation; training itself never waits like this). GPU: a one-thread kernel on the compute
        stream spins on the locally written acknowledgement words, the host just synchronises the stream."""
        if self.cfg.backend == "cuda":
            self._serve_local()
            self.drain()
            if self.cfg.push_mode != "mailbox" or not self.inbox_order or (self._exec is None and self._fexec is None):
                return
            stream = self.compute_stream
            N.check(self.lib.dm_launch_wait_ack(self.seg.addr("inbox"), len(self.inbox_order), self._seq_word_ptr(),
                                                stream), "wait_ack")
            N.check(self.lib.dm_stream_sync(stream), "wait for the ps acknowledgements")
            return
        if self.cfg.push_mode != "mailbox" or not self.inbox_order:
            return
        seq = self._seq_host
        t0 = time.time()
        while True:
            inbox = self._read_own("inbox", 2 * len(self.inbox_order))
            if all(((inbox[2 * i] - seq) & 0xFFFFFFFF) < 0x80000000 for i in range(len(self.inbox_order))):
                return
            if time.time() - t0 > timeout_s:
                raise TimeoutError(f"pushes up to {seq} not acknowledged: inbox={inbox}")
            time.sleep(0.0002)

    def attach_local_ps(self, ps_list) -> None:
        """In-process clusters whose ps tasks run in one-shot mode: after every launch of step kernels the worker
        lets those ps tasks run their serve kernel once (stream-ordered behind the steps)."""
        self._ps_local = [p for p in ps_list if getattr(p, "oneshot", False)]

    def _serve_local(self) -> None:
        if self._ps_local and (self._exec or self._fexec):
            stream = self.compute_stream
            for p in self._ps_local:
                p.serve_once(after_stream=stream, wait=True)

    def heartbeat(self) -> None:
        """Liveness mark for the ps-side failure detector (`ParameterServer.join(worker_timeout_s=...)`)."""
        self.rdv.put(f"session/heartbeat/{self.task_index}", time.time())

    def _start_heartbeat_thread(self, period_s: float = 0.5) -> None:
        """Process-level liveness: a daemon thread with its own store connection refreshes the heartbeat twice a
        second for as long as this process lives (a crash, `os._exit` or `kill -9` silences it at once), so a worker
        that is merely busy — graph capture, a long chunk of steps on a loaded box, waiting for the chief — is never
        mistaken for a dead one, however small `--worker_timeout` is."""
        if getattr(self, "_hb_thread", None) is not None:
            return
        import threading

        self._hb_stop = threading.Event()
        key = f"session/heartbeat/{self.task_index}"

        def loop():
            try:
                rdv = self.rdv.clone()
            except Exception:
                return
            while not self._hb_stop.wait(period_s):
                try:
                    rdv.put(key, time.time())
                except Exception:
                    return      # the store is gone: the session is over

        self._hb_thread = threading.Thread(target=loop, name="dm-heartbeat", daemon=True)
        self._hb_thread.start()

    @nvtx_annotate("dm.worker.prepare")
    def prepare(self) -> None:
        """Build the step graphs (GPU backend). Only needs the PS pointers, so it may run before the variables
        are initialised — in-process clusters call it before the persistent PS kernel is launched so that no
        allocation happens while that kernel owns part of the GPU."""
        if self.cfg.backend == "cuda" and self._exec is None and self._fexec is None:
            if self.engine == "fused":
                self._build_fused()
            else:
                self._build_cuda()

    # ------------------------------------------------------------------------------------------
    # variable I/O through peer memory (chief init / restore, checkpoints, evaluation)
    # ------------------------------------------------------------------------------------------
    def _copy_to_ps(self, k: int, region: str, elem_offset: int, src: torch.Tensor) -> None:
        src = src.contiguous()
        nbytes = src.numel() * src.element_size()
        dst = self.ps_segs[k].addr(region, elem_offset * src.element_size())
        if self.cfg.backend == "cuda":
            host = src.cpu()
            N.check(self.lib.dm_memcpy_async(dst, host.data_ptr(), nbytes, None), "copy to ps")
            N.check(self.lib.dm_stream_sync(None))
        else:
            C.memmove(dst, src.data_ptr(), nbytes)

    def _copy_from_ps(self, k: int, region: str, elem_offset: int, count: int, dtype: torch.dtype) -> torch.Tensor:
        out = torch.empty(count, dtype=dtype)
        nbytes = count * out.element_size()
        src = self.ps_segs[k].addr(region, elem_offset * out.element_size())
        if self.cfg.backend == "cuda":
            N.check(self.lib.dm_memcpy_async(out.data_ptr(), src, nbytes, None), "copy from ps")
            N.check(self.lib.dm_stream_sync(None))
        else:
            C.memmove(out.data_ptr(), src, nbytes)
        return out

    def _pack(self, vl: VarLayout, t: torch.Tensor) -> torch.Tensor:
        """Variable tensor ([out, in] or [out]) -> arena span (row padding applied)."""
        t = t.detach().to(torch.float32).cpu()
        if t.dim() == 2 and vl.ld != vl.cols:
            buf = torch.zeros(vl.rows, vl.ld)
            buf[:, :vl.cols] = t
            return buf.reshape(-1)
        return t.reshape(-1).contiguous()

    def _unpack(self, vl: VarLayout, flat: torch.Tensor) -> torch.Tensor:
        if len(vl.spec.shape) == 2:
            return flat.view(vl.rows, vl.ld)[:, :vl.cols].clone()
        return flat.clone()

    def write_variables(self, params: Dict[str, torch.Tensor], region: str = "params") -> None:
        for name, t in params.items():
            vl = self.layout.by_name[name]
            if tuple(t.shape) != tuple(vl.spec.shape):
                raise ValueError(f"{name}: expected shape {vl.spec.shape}, got {tuple(t.shape)}")
            flat = self._pack(vl, t)
            # a column-split variable keeps its full span on every owning shard (each shard updates its own columns)
            for k, off in dict.fromkeys((pc.ps, pc.offset) for pc in vl.pieces):
                self._copy_to_ps(k, region, off, flat)
                if region == "params" and self.cfg.dtype == "bf16":
                    self._copy_to_ps(k, "shadow", off, flat.to(torch.bfloat16))

    def read_variables(self, region: str = "params") -> Dict[str, torch.Tensor]:
        out = {}
        for name, vl in self.layout.by_name.items():
            if len({(pc.ps, pc.offset) for pc in vl.pieces}) == 1:   # one owner (whole variable, or all slices there)
                flat = self._copy_from_ps(vl.ps, region, vl.offset, vl.span, torch.float32)
                out[name] = self._unpack(vl, flat)
                continue
            full = torch.empty(vl.rows, vl.cols)
            cache: Dict[Tuple[int, int], torch.Tensor] = {}
            for pc in vl.pieces:
                if pc.c1 <= pc.c0:
                    continue
                if (pc.ps, pc.offset) not in cache:
                    cache[(pc.ps, pc.offset)] = self._unpack(
                        vl, self._copy_from_ps(pc.ps, region, pc.offset, vl.span, torch.float32))
                full[:, pc.c0:pc.c1] = cache[(pc.ps, pc.offset)][:, pc.c0:pc.c1]
            out[name] = full
        return out

    def read_global_step(self) -> int:
        t = self._copy_from_ps(self.gs_owner, "ctrl", CTRL_GLOBAL_STEP, 1, torch.int32)
        return int(t.item()) & 0xFFFFFFFF

    def write_global_step(self, value: int) -> None:
        self._copy_to_ps(self.gs_owner, "ctrl", CTRL_GLOBAL_STEP, torch.tensor([value], dtype=torch.int32))

    def read_item_state(self, k: int) -> torch.Tensor:
        ni = max(self.layout.shards[k].n_items, 1)
        return self._copy_from_ps(k, "item_state", 0, ni * 4, torch.int32)

    def write_item_state(self, k: int, state: torch.Tensor) -> None:
        self._copy_to_ps(k, "item_state", 0, state.to(torch.int32))

    @nvtx_annotate("dm.worker.initialize_variables")
    def initialize_variables(self, seed: int = 0, params: Optional[Dict[str, torch.Tensor]] = None) -> None:
        """Chief-only: run the initialisers on the PS shards and announce `init/done` (DS:108-109)."""
        if not self.is_chief:
            raise RuntimeError("only the chief (worker 0) initialises variables")
        params = params if params is not None else mlp.init_params(self.spec, seed)
        self.write_variables(params)
        zeros = {k: torch.zeros_like(v) for k, v in params.items()}
        self.write_variables(zeros, "adam_m")
        self.write_variables(zeros, "adam_v")
        self.rdv.put("init/done", {"seed": seed, "by": self.task_index})

    def variables_are_live(self) -> bool:
        """True when some chief incarnation has already initialised (or restored) the variables on the ps tasks of
        this session. A restarted chief must then *not* run the initialisers again: the shards keep training state
        (parameters, Adam slots, per-item step counts, global_step) that the other workers are still updating."""
        return self.rdv.try_get("init/done") is not None

    def mark_initialized(self) -> None:
        """Chief-only: announce that the variables on the PS are valid (after a checkpoint restore)."""
        self.rdv.put("init/done", {"restored": True, "by": self.task_index})

    # ------------------------------------------------------------------------------------------
    # GPU step construction
    # ------------------------------------------------------------------------------------------
    def _push_target(self, k: int, seq_ptr: int) -> N.PushTarget:
        seg, desc = self.ps_segs[k], self.ps_desc[k]
        t = N.PushTarget()
        w = self.task_index
        arena, ni, ns = desc["arena_elems"], max(desc.get("n_flags", desc["n_items"]), 1), self.cfg.nslots
        if self.cfg.push_mode == "atomic":
            t.mode, t.scale, t.base = N.PUSH_ATOMIC, -self.opt.lr, seg.addr("params")
            t.nslots = 1
        else:
            t.mode, t.scale = N.PUSH_MAILBOX, 1.0
            t.base = seg.addr("mailbox", w * ns * arena * 4)
            t.slot_stride = arena
            t.flags = seg.addr("flags", w * ns * ni * 4)
            t.flag_slot_stride = ni
            t.nslots = ns
        t.seq_ptr = seq_ptr
        # ps shard on our own GPU (in-process / colocated): gpu-scope release suffices for its flags
        t.gpu_scope = int(self.cfg.backend == "cuda" and desc.get("device", -2) == self.device
                          and self.cluster.num_workers == 1)
        return t

    def _weight_ptr(self, vl: VarLayout) -> int:
        seg = self.ps_segs[vl.ps]
        if self.cfg.dtype == "bf16":
            return seg.addr("shadow", vl.offset * 2)
        return seg.addr("params", vl.offset * 4)

    def _build_cuda(self) -> None:
        spec, cfg, lay = self.spec, self.cfg, self.layout
        N.ensure_prepared(self.device)
        x_bytes = self.B_pad * self.ld_in * self.es
        y_bytes = self.B_pad * spec.num_classes * 4
        out = C.c_void_p()
        N.check(self.lib.dm_exec_create(self.device, cfg.ring_slots, cfg.lanes, cfg.graph_steps, x_bytes, y_bytes,
                                        C.byref(out)), "exec create")
        self._exec = out.value
        self.x_bytes, self.y_bytes = x_bytes, y_bytes
        dev = f"cuda:{self.device}"
        names = spec.variable_names()
        sizes = spec.layer_sizes
        L = len(sizes)
        # activations / pre-activation gradients of the hidden layers (row padded, zero initialised)
        # (one set per executor slot: steps of different slots may run concurrently)
        self._slot_act = [[None] + [torch.zeros(self.B_pad, gemm_ops.padded_ld(sizes[l][1]), dtype=self.tdtype,
                                                device=dev) for l in range(L - 1)] for _ in range(cfg.ring_slots)]
        self._slot_dact = [[None] + [torch.zeros_like(a[l + 1]) for l in range(L - 1)] for a in self._slot_act]
        self.act, self.dact = self._slot_act[0], self._slot_dact[0]
        seq_counter = self.seg.addr("seq")
        self._slots = []
        stream = self.lib.dm_exec_compute_stream(self._exec)
        # ---- evaluation path (forward + head without gradients; shares the activation buffers) ----
        self._eval_x = torch.zeros(self.B_pad, self.ld_in, dtype=self.tdtype, device=dev)
        self._eval_y = torch.zeros(self.B_pad, spec.num_classes, dtype=torch.float32, device=dev)
        self._eval_res = torch.zeros(4, dtype=torch.int32, device=dev)
        self._eval_plans = []
        for l in range(L - 1):
            wl, bl = lay.by_name[names[l][0]], lay.by_name[names[l][1]]
            fin, fout = sizes[l]
            self._eval_plans.append(gemm_ops.forward_plan(
                w_ptr=self._weight_ptr(wl), x_ptr=self._eval_x.data_ptr() if l == 0 else self.act[l].data_ptr(),
                out_ptr=self.act[l + 1].data_ptr(), bias_ptr=self.ps_segs[bl.ps].addr("params", bl.offset * 4),
                O=fout, I=fin, B=self.batch, B_pad=self.B_pad, dtype=self.dt, relu=True, ldw=wl.ld,
                ldx=self.ld_in if l == 0 else self.act[l].shape[1], ldo=self.act[l + 1].shape[1], name=f"eval_fwd{l}"))
        wl, bl = lay.by_name[names[L - 1][0]], lay.by_name[names[L - 1][1]]
        self._eval_plans.append(head_ops.head_plan(
            h_ptr=self.act[L - 1].data_ptr(), labels_ptr=self._eval_y.data_ptr(),
            w_last_ptr=self.ps_segs[wl.ps].addr("params", wl.offset * 4),
            b_last_ptr=self.ps_segs[bl.ps].addr("params", bl.offset * 4), dpre_ptr=self.dact[L - 1].data_ptr(),
            result_ptr=self._eval_res.data_ptr(), B=self.batch, B_pad=self.B_pad, H=sizes[L - 1][0],
            num_classes=spec.num_classes, loss_kind=N.LOSS_BOOK if spec.loss == "book" else N.LOSS_XENT,
            act_bf16=cfg.dtype == "bf16", compute_grads=False, ldh=self.act[L - 1].shape[1]))
        torch.cuda.synchronize(self.device)
        for slot in range(cfg.ring_slots):
            act, dact = self._slot_act[slot], self._slot_dact[slot]
            seq_ptr = self.seg.addr("seq", 4 * (1 + slot))
            stream = self.lib.dm_exec_capture_stream(self._exec, slot)
            xd, yd, rd, xs, ys = (C.c_void_p() for _ in range(5))
            N.check(self.lib.dm_exec_slot_info(self._exec, slot, C.byref(xd), C.byref(yd), C.byref(rd), C.byref(xs),
                                               C.byref(ys)))
            plans = []
            # ---- forward: hidden layers, W pulled from the PS shard by TMA ----
            for l in range(L - 1):
                wn, bn = names[l]
                wl, bl = lay.by_name[wn], lay.by_name[bn]
                fin, fout = sizes[l]
                in_ptr = xd.value if l == 0 else act[l].data_ptr()
                ld_in = self.ld_in if l == 0 else act[l].shape[1]
                plans.append(gemm_ops.forward_plan(
                    w_ptr=self._weight_ptr(wl), x_ptr=in_ptr, out_ptr=act[l + 1].data_ptr(),
                    bias_ptr=self.ps_segs[bl.ps].addr("params", bl.offset * 4), O=fout, I=fin, B=self.batch,
                    B_pad=self.B_pad, dtype=self.dt, relu=True, ldw=wl.ld, ldx=ld_in, ldo=act[l + 1].shape[1],
                    bump_seq_ptr=seq_ptr if l == 0 else 0, seq_counter_ptr=seq_counter, name=f"fwd{l}"))
            # ---- classifier head ----
            wn, bn = names[L - 1]
            wl, bl = lay.by_name[wn], lay.by_name[bn]
            hb = lay.by_name[names[L - 2][1]]  # bias of the last hidden layer
            inbox_ptr = self.seg.addr("inbox") if cfg.push_mode == "mailbox" else 0
            gs_ptr = self.ps_segs[self.gs_owner].addr("ctrl", 4 * CTRL_GLOBAL_STEP) if cfg.push_mode == "atomic" else 0
            head = head_ops.head_plan(
                h_ptr=act[L - 1].data_ptr(), labels_ptr=yd.value,
                w_last_ptr=self.ps_segs[wl.ps].addr("params", wl.offset * 4),
                b_last_ptr=self.ps_segs[bl.ps].addr("params", bl.offset * 4),
                dpre_ptr=dact[L - 1].data_ptr(), result_ptr=rd.value, B=self.batch, B_pad=self.B_pad,
                H=sizes[L - 1][0], num_classes=spec.num_classes,
                loss_kind=N.LOSS_BOOK if spec.loss == "book" else N.LOSS_XENT, act_bf16=cfg.dtype == "bf16",
                push=self._push_target(wl.ps, seq_ptr), push_bh=self._push_target(hb.ps, seq_ptr),
                push_bl=self._push_target(bl.ps, seq_ptr),
                off_w_last=wl.offset, off_b_last=bl.offset, off_b_hidden=hb.offset,
                item_w_last_base=wl.item_base, item_b_last=bl.item_base, item_b_hidden_base=hb.item_base,
                seq_ptr=seq_ptr, inbox_ptr=inbox_ptr, n_inbox=len(self.inbox_order), ps_global_step_ptr=gs_ptr,
                nslots=cfg.nslots, ldh=act[L - 1].shape[1])
            plans.append(head)
            # ---- backward of the hidden layers: dX (+ bias-grad push) *before* dW (fused push) of the same layer:
            #      dX pulls W_l from the PS a second time, and the PS applies a pushed dW_l within microseconds,
            #      so pushing dW_l first would let this step's own update leak into its dX ----
            for l in range(L - 2, -1, -1):
                wn, bn = names[l]
                wl = lay.by_name[wn]
                fin, fout = sizes[l]
                in_ptr = xd.value if l == 0 else act[l].data_ptr()
                ld_in = self.ld_in if l == 0 else act[l].shape[1]
                if l > 0:
                    pb = lay.by_name[names[l - 1][1]]  # bias of the previous hidden layer gets its grad here
                    plans.append(gemm_ops.dx_plan(
                        w_ptr=self._weight_ptr(wl), dy_ptr=dact[l + 1].data_ptr(), out_ptr=dact[l].data_ptr(),
                        mask_ptr=act[l].data_ptr(), O=fout, I=fin, B=self.batch, B_pad=self.B_pad, dtype=self.dt,
                        ldw=wl.ld, lddy=dact[l + 1].shape[1], ldo=dact[l].shape[1],
                        colsum=self._push_target(pb.ps, seq_ptr), colsum_offset=pb.offset, colsum_item_base=pb.item_base,
                        name=f"dx{l}"))
                plans.append(gemm_ops.dw_plan(
                    dy_ptr=dact[l + 1].data_ptr(), x_ptr=in_ptr, O=fout, I=fin, B_pad=self.B_pad, dtype=self.dt,
                    push=self._push_target(wl.ps, seq_ptr), push_offset=wl.offset, item_base=wl.item_base,
                    bn=lay.dw_tile_n, lddy=dact[l + 1].shape[1], ldx=ld_in, ldw=wl.ld, name=f"dw{l}"))
            if cfg.pdl:
                # programmatic dependent launch inside the step graph: kernel k+1's prologue (and the head's
                # W_last fetch) overlaps kernel k; every kernel waits on griddepcontrol.wait before it touches
                # its predecessor's outputs. The first kernel keeps a full dependency on the previous step.
                for p in plans[1:]:
                    p.params.pdl = 1
            self.kernels_per_step = len(plans)
            N.check(self.lib.dm_exec_begin_capture(self._exec, slot), "begin capture")
            try:
                for p in plans:
                    p.launch(stream)
            finally:
                N.check(self.lib.dm_exec_end_capture(self._exec, slot, len(plans)), "end capture")
            x_stage = torch.from_numpy(np.frombuffer((C.c_uint8 * x_bytes).from_address(xs.value), dtype=np.uint8))
            y_stage = torch.from_numpy(np.frombuffer((C.c_uint8 * y_bytes).from_address(ys.value), dtype=np.uint8))
            self._slots.append({
                "plans": plans, "x_dev": xd.value, "y_dev": yd.value, "res_dev": rd.value,
                "x_stage": x_stage.view(self.tdtype).view(self.B_pad, self.ld_in), "x_stage_ptr": xs.value,
                "y_stage": y_stage.view(torch.float32).view(self.B_pad, spec.num_classes), "y_stage_ptr": ys.value,
            })

        # group graphs: the U steps of a group as parallel chains of one graph (native loops launch these)
        U = cfg.graph_steps
        if U > 1:
            for g in range(cfg.ring_slots // U):
                N.check(self.lib.dm_exec_begin_group_capture(self._exec, g), "begin group capture")
                try:
                    for u in range(U):
                        slot = g * U + u
                        st = self.lib.dm_exec_capture_stream(self._exec, slot)
                        for p in self._slots[slot]["plans"]:
                            p.launch(st)
                finally:
                    N.check(self.lib.dm_exec_end_group_capture(self._exec, g), "end group capture")

    # ------------------------------------------------------------------------------------------
    # fused engine construction
    # ------------------------------------------------------------------------------------------
    def _fused_maps(self, x_ptr: int, n_rows: int) -> N.FusedMaps:
        """Tensor maps of one fused launch: W K-slices on the owning shards (NVLink peer mappings) and the two views
        of the x matrix [n_rows][in] the batches are taken from."""
        lay, I = self.layout, self.spec.in_features
        wname = self.spec.variable_names()[0][0]
        vl = lay.by_name[wname]
        m = N.FusedMaps()
        for sl in lay.fused_slices:
            seg = self.ps_segs[sl.ps]
            tm = N.make_tensor_map(seg.addr("params", sl.w_offset * 4), N.DT_F32, I, vl.rows, vl.ld * 4, 32, 128)
            C.memmove(C.addressof(m.w[sl.rank]), C.addressof(tm), N.TENSOR_MAP_BYTES)
            # destination of this CTA's TMA-store push: [slot][H][I] view of our mailbox for the hidden weight on that
            # shard (mailbox mode), or of the master copy itself (atomic mode: TMA reduce-add, push == apply)
            desc = self.ps_desc[sl.ps]
            arena, ns = desc["arena_elems"], self.cfg.nslots
            if self.cfg.push_mode == "atomic":
                tp = N.make_tensor_map_3d(seg.addr("params", sl.w_offset * 4), I, vl.rows, 1, vl.ld * 4, arena * 4, 32, 128)
            else:
                base = seg.addr("mailbox", (self.task_index * ns * arena + sl.w_offset) * 4)
                tp = N.make_tensor_map_3d(base, I, vl.rows, ns, vl.ld * 4, arena * 4, 32, 128)
            C.memmove(C.addressof(m.push[sl.rank]), C.addressof(tp), N.TENSOR_MAP_BYTES)
        xk = N.make_tensor_map(x_ptr, N.DT_F32, I, n_rows, I * 4, 32, 32)
        xmn = N.make_tensor_map(x_ptr, N.DT_F32, I, n_rows, I * 4, 32, 32, mn_major=True)
        C.memmove(C.addressof(m.xk), C.addressof(xk), N.TENSOR_MAP_BYTES)
        C.memmove(C.addressof(m.xmn), C.addressof(xmn), N.TENSOR_MAP_BYTES)
        return m

    def _build_fused(self) -> None:
        spec, cfg, lay = self.spec, self.cfg, self.layout
        N.ensure_prepared(self.device)
        I, H = spec.layer_sizes[0]
        Cn = spec.num_classes
        max_lanes = C.c_int(0)
        N.check(self.lib.dm_fused_max_lanes(self.device, C.byref(max_lanes)), "fused occupancy")
        lanes = max(1, min(cfg.lanes, max_lanes.value if max_lanes.value > 0 else cfg.lanes))
        self.fused_lanes = lanes
        if "DM_GATHER_THREADS" not in os.environ:
            # the gather pool spins while a run is active: share the host's cores between the worker processes of
            # this node (torchrun exports LOCAL_WORLD_SIZE; a stand-alone task assumes it has the node to itself)
            local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
            # Measured on the 4-GPU boxes (48-core quota, 3 workers): 5 helpers per worker -> 398 k steps/s host-fed,
            # 9 or 12 -> 137-153 k (CFS throttling: NCCL's proxy threads, the clock sampler and the interpreters
            # spend quota too). A single process on a node (quota 16 on the 1-GPU boxes) does best with 12.
            cores = usable_cores()
            n = min(12, cores - 3) if local_world == 1 else min(8, cores // (2 * local_world) - 1)
            os.environ["DM_GATHER_THREADS"] = str(max(2, n))
        out = C.c_void_p()
        N.check(self.lib.dm_fexec_create(self.device, lanes, I, Cn, self.batch, C.byref(out)), "fused exec create")
        self._fexec = out.value
        xd, yd, xs, ys, ctl = (C.c_void_p() for _ in range(5))
        slots = C.c_int(0)
        N.check(self.lib.dm_fexec_buffers(self._fexec, C.byref(xd), C.byref(yd), C.byref(xs), C.byref(ys),
                                          C.byref(ctl), C.byref(slots)))
        self._fx_x_dev, self._fx_y_dev, self._fx_ctl, self._fx_slots = xd.value, yd.value, ctl.value, slots.value
        self.x_bytes = N.FUSED_ROWS_PER_SLOT * I * 4
        self.y_bytes = N.FUSED_ROWS_PER_SLOT * Cn * 4
        names = spec.variable_names()
        hb, wl, bl = lay.by_name[names[0][1]], lay.by_name[names[1][0]], lay.by_name[names[1][1]]
        hw = lay.by_name[names[0][0]]
        p = N.FusedParams()
        p.B, p.H, p.C, p.I = self.batch, H, Cn, I
        p.loss_kind = N.LOSS_BOOK if spec.loss == "book" else N.LOSS_XENT
        p.ldw = hw.ld
        p.strict = int(cfg.strict_steps)
        # shards this worker pushes to, the global-step owner first (same order as the inbox entries)
        order = list(self.inbox_order)
        for k in range(self.cluster.num_ps):       # atomic mode has no inbox: every shard with items, in order
            if k not in order and lay.shards[k].n_items > 0:
                order.append(k)
        if len(order) > N.FUSED_MAX_SHARDS:
            raise ValueError(f"the fused engine talks to at most {N.FUSED_MAX_SHARDS} ps shards")
        sidx = {k: i for i, k in enumerate(order)}
        p.n_shards = len(order)
        for i, k in enumerate(order):
            p.shard[i].push = self._push_target(k, 0)
            p.shard[i].inbox = (self.seg.addr("inbox", 8 * self.inbox_index[k])
                                if (cfg.push_mode == "mailbox" and k in self.inbox_index) else None)
        for sl in lay.fused_slices:
            fs = p.slice[sl.rank]
            fs.kc_begin, fs.kc_count, fs.shard, fs.flag_index, fs.w_offset = (sl.kc_begin, sl.kc_count, sidx[sl.ps],
                                                                               sl.flag, sl.w_offset)
        p.bias_h = self.ps_segs[hb.ps].addr("params", hb.offset * 4)
        p.w_last = self.ps_segs[wl.ps].addr("params", wl.offset * 4)
        p.b_last = self.ps_segs[bl.ps].addr("params", bl.offset * 4)
        p.shard_bh, p.shard_wl, p.shard_bl = sidx[hb.ps], sidx[wl.ps], sidx[bl.ps]
        p.flag_bh, p.flag_wl, p.flag_bl = hb.flag_base, wl.flag_base, bl.flag_base
        p.off_bh, p.off_wl, p.off_bl = hb.offset, wl.offset, bl.offset
        p.y_base = self._fx_y_dev
        p.row_start, p.row_stride, p.row_wrap = 0, N.FUSED_ROWS_PER_SLOT, self._fx_slots * N.FUSED_ROWS_PER_SLOT
        p.nslots = cfg.nslots
        p.ps_global_step = (self.ps_segs[self.gs_owner].addr("ctrl", 4 * CTRL_GLOBAL_STEP)
                            if cfg.push_mode == "atomic" else None)
        if os.environ.get("DM_FUSED_DEBUG_TS") == "1":
            self._fx_dbg = torch.zeros(64, dtype=torch.int64, device=f"cuda:{self.device}")
            p.debug_ts = self._fx_dbg.data_ptr()
        self._fx_params = p
        self._fx_maps = self._fused_maps(self._fx_x_dev, self._fx_slots * N.FUSED_ROWS_PER_SLOT)
        N.check(self.lib.dm_fexec_set_params(self._fexec, C.addressof(self._fx_maps), C.addressof(p)), "set params")
        self._fx_ds_maps: Dict[Tuple[int, int], N.FusedMaps] = {}
        self._fx_stage_x = torch.zeros(1, N.FUSED_ROWS_PER_SLOT, I, dtype=torch.float32)
        self._fx_stage_y = torch.zeros(1, N.FUSED_ROWS_PER_SLOT, Cn, dtype=torch.float32)
        self._fx_tickets: Dict[int, StepOutput] = {}
        self._fx_ticket = 0
        # evaluation buffers (allocated now: nothing is allocated once a persistent ps kernel may be resident)
        self._ev_rows = 4096
        self._ev_dev = torch.zeros(2 * self._ev_rows, Cn, dtype=torch.float32, device=f"cuda:{self.device}")
        self._ev_cnt = torch.zeros(1, dtype=torch.int32, device=f"cuda:{self.device}")
        self._ev_pin = torch.zeros(2 * self._ev_rows, Cn, dtype=torch.float32).pin_memory()
        self._ev_cnt_pin = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.kernels_per_step = 1
        torch.cuda.synchronize(self.device)

    # ------------------------------------------------------------------------------------------
    # stepping
    # ------------------------------------------------------------------------------------------
    def submit(self, x: torch.Tensor, y: torch.Tensor) -> int:
        """Enqueue one training step on a host batch (x [B, in] float, y [B, classes] one-hot). Returns a ticket."""
        if self.cfg.backend != "cuda":
            raise RuntimeError("submit/result pipelining exists on the cuda backend; use step() on cpu")
        if self.engine == "fused":
            # the fused engine pipelines *inside* run_steps (chunks); a single submitted step runs to completion
            out = self._fused_steps_host(x, y)
            self._fx_ticket += 1
            self._fx_tickets[self._fx_ticket] = out
            if len(self._fx_tickets) > 4096:
                self._fx_tickets.pop(next(iter(self._fx_tickets)))
            return self._fx_ticket
        slot = C.c_int()
        N.check(self.lib.dm_exec_acquire_slot(self._exec, C.byref(slot)), "acquire slot")
        s = self._slots[slot.value]
        b = x.shape[0]
        if b != self.batch:
            raise ValueError(f"expected a batch of {self.batch}, got {b}")
        s["x_stage"][:b, :x.shape[1]].copy_(x)
        s["y_stage"][:b].copy_(y)
        t = C.c_uint64()
        N.check(self.lib.dm_exec_submit(self._exec, s["x_stage_ptr"], s["y_stage_ptr"], C.byref(t)), "submit")
        return t.value

    def set_lanes(self, lanes: int, strict: Optional[bool] = None) -> None:
        """Fused engine: change the number of steps in flight (clusters per launch) and, optionally, the strict
        read-your-writes pull order — e.g. `set_lanes(1, strict=True)` is the reference's sequential worker loop."""
        if self.engine != "fused" or not self._fexec:
            raise RuntimeError("set_lanes applies to a prepared fused engine")
        if lanes < 1 or (self.cfg.push_mode == "mailbox" and lanes > self.cfg.nslots):
            raise ValueError("lanes must be in [1, nslots]")
        self.drain()
        N.check(self.lib.dm_fexec_set_lanes(self._fexec, lanes), "set lanes")
        self.fused_lanes = lanes
        if strict is not None:
            self._fx_params.strict = int(strict)
            N.check(self.lib.dm_fexec_set_params(self._fexec, C.addressof(self._fx_maps), C.addressof(self._fx_params)),
                    "set params")

    def _fused_steps_host(self, x: torch.Tensor, y: torch.Tensor) -> StepOutput:
        b = x.shape[0]
        if b != self.batch:
            raise ValueError(f"expected a batch of {self.batch}, got {b}")
        self._fx_stage_x[0, :b].copy_(x.reshape(b, -1))
        self._fx_stage_y[0, :b].copy_(y)
        r = N.StepResult()
        done = C.c_uint32(0)
        N.check(self.lib.dm_fexec_steps_host(self._fexec, self._fx_stage_x.data_ptr(), self._fx_stage_y.data_ptr(), 1,
                                             C.addressof(r), C.byref(done)), "fused step")
        if done.value != 1:
            raise N.NativeError("fused step did not run")
        self._serve_local()
        return StepOutput(r.loss, r.global_step, r.correct, r.seq)

    def submit_resident(self, x_ptr: int = 0, y_ptr: int = 0) -> int:
        """Enqueue a step whose inputs already live in device (or pinned) memory at x_ptr / y_ptr, laid out
        exactly like the slot buffers ([B_pad][ld_in] compute dtype, [B_pad][classes] fp32). 0 = reuse the
        data already in the slot."""
        t = C.c_uint64()
        N.check(self.lib.dm_exec_submit(self._exec, x_ptr or None, y_ptr or None, C.byref(t)), "submit")
        return t.value

    def run_resident(self, n_steps: int, x_base_ptr: int, y_base_ptr: int, x_row_bytes: int, y_row_bytes: int,
                     n_rows: int, start: int = 0, wait_applied: bool = False, timed: bool = False) -> None:
        """Native loop over a device-resident dataset: step i trains on rows ((start + i) * batch) % n_rows ..
        (contiguous). Graph engine: copied device-to-device into the slot buffers; fused engine: one launch whose
        TMA loads read the rows straight out of the dataset. Results stay in the executor."""
        if self.engine == "fused":
            if x_row_bytes != self.spec.in_features * 4 or y_row_bytes != self.spec.num_classes * 4:
                raise ValueError("fused run_resident: dataset rows must be dense fp32 [in] / [classes]")
            key = (x_base_ptr, n_rows)
            if key not in self._fx_ds_maps:
                self._fx_ds_maps[key] = self._fused_maps(x_base_ptr, n_rows + N.FUSED_ROWS_PER_SLOT)
            # wait_applied: the launch itself ends with the wait for the ps acknowledgement of its last push (no extra
            # kernel); only meaningful when a persistent ps kernel is serving
            wa = int(wait_applied and not self._ps_local)
            N.check(self.lib.dm_fexec_run_resident(self._fexec, C.addressof(self._fx_ds_maps[key]), y_base_ptr,
                                                   start * self.batch, self.batch, n_rows, n_steps, wa, int(timed)),
                    "run resident")
            self._serve_local()
            return
        N.check(self.lib.dm_exec_run_resident(self._exec, n_steps, x_base_ptr, y_base_ptr, x_row_bytes, y_row_bytes,
                                              n_rows, self.batch, start), "run resident")

    def last_resident_result(self) -> StepOutput:
        """Result of the final step of the most recent `run_resident` (waits for it)."""
        if self.engine == "fused":
            n = C.c_uint64()
            N.check(self.lib.dm_fexec_resident_results(self._fexec, None, 2 ** 64 - 1, C.byref(n)), "resident results")
            if n.value == 0:
                raise N.NativeError("no resident run to report on")
            res = (N.StepResult * n.value)()
            N.check(self.lib.dm_fexec_resident_results(self._fexec, C.addressof(res), n.value, C.byref(n)),
                    "resident results")
            r = res[n.value - 1]
            return StepOutput(r.loss, r.global_step, r.correct, r.seq)
        return self.result(int(self.lib.dm_exec_submitted(self._exec)), wait=True)

    def last_elapsed_ms(self) -> float:
        """Fused engine: device time (CUDA events recorded natively right around the launch) of the most recent
        `run_resident(..., timed=True)`."""
        ms = C.c_float(0.0)
        N.check(self.lib.dm_fexec_last_elapsed_ms(self._fexec, C.byref(ms)), "elapsed")
        return float(ms.value)

    def result(self, ticket: int, wait: bool = True) -> Optional[StepOutput]:
        if self.engine == "fused" and self.cfg.backend == "cuda":
            return self._fx_tickets[ticket]
        r = N.StepResult()
        rc = self.lib.dm_exec_result(self._exec, ticket, C.addressof(r), int(wait))
        if rc == 1:
            return None
        if rc != 0:
            N.check(rc if rc < 0 else -rc, "result")
        return StepOutput(r.loss, r.global_step, r.correct, r.seq)

    def step(self, x: torch.Tensor, y: torch.Tensor) -> StepOutput:
        """One synchronous training step — the analogue of `sess.run([train_op, loss, global_step], feed_dict)`."""
        if self.cfg.backend == "cuda":
            if self.engine == "fused":
                return self._fused_steps_host(x, y)
            out = self.result(self.submit(x, y), wait=True)
            self._serve_local()
            return out
        return self._cpu_step(x, y)

    def make_loader(self, images: torch.Tensor, labels: torch.Tensor, seed: int = 0, shuffle: bool = True,
                    epoch_feed: Optional[bool] = None):
        """Native `next_batch` loader over a host dataset (kept alive by the returned object)."""
        return NativeLoader(self, images, labels, seed, shuffle, epoch_feed)

    def feed_stats(self) -> Dict[str, int]:
        """Fused executor: chunks fed straight from the loader's epoch buffer / through the row gather, epoch fills
        handed to the helper threads (all zero on other engines)."""
        if not self._fexec:
            return {"direct_chunks": 0, "gathered_chunks": 0, "fills_posted": 0}
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self.lib.dm_fexec_feed_stats(self._fexec, C.byref(a), C.byref(b), C.byref(c))
        return {"direct_chunks": int(a.value), "gathered_chunks": int(b.value), "fills_posted": int(c.value)}

    @nvtx_annotate("dm.worker.run_steps")
    def run_steps(self, n_steps: int, loader: "NativeLoader", stop_at_global_step: int = 0,
                  wait_applied: bool = False) -> Sequence[StepOutput]:
        """Native train loop: n_steps x (next_batch -> H2D -> step kernels -> result D2H). `wait_applied`: return only
        once every push of the run has been applied by the ps tasks (fused engine: the tail of the last launch waits
        for the acknowledgements; otherwise `wait_applied()` is called)."""
        if self.cfg.backend != "cuda":
            out = []
            for _ in range(n_steps):
                x, y = loader.next_batch()
                r = self._cpu_step(x, y)
                out.append(r)
                if stop_at_global_step and r.global_step >= stop_at_global_step:
                    break
            if wait_applied:
                self.wait_applied()
            return out
        res = (N.StepResult * n_steps)()
        done = C.c_uint64()
        if self.engine == "fused":
            in_kernel = wait_applied and not stop_at_global_step and not self._ps_local
            N.check(self.lib.dm_fexec_run(self._fexec, loader.handle, n_steps, C.addressof(res), stop_at_global_step,
                                          C.byref(done), int(in_kernel)), "fused exec run")
            if in_kernel:
                wait_applied = False
        else:
            N.check(self.lib.dm_exec_run(self._exec, loader.handle, n_steps, C.addressof(res), stop_at_global_step,
                                         C.byref(done)), "exec run")
        self._serve_local()
        if wait_applied:
            self.wait_applied()
        raw = np.frombuffer(res, dtype=_STEP_DTYPE, count=n_steps)[: done.value]   # keeps `res` alive
        return StepOutputs(raw)

    def drain(self) -> None:
        if self._fexec:
            N.check(self.lib.dm_fexec_drain(self._fexec), "drain")
        if self._exec:
            N.check(self.lib.dm_exec_drain(self._exec), "drain")

    @property
    def compute_stream(self) -> int:
        """Raw cudaStream_t of the executor's compute stream (for CUDA-event timing of a run of steps)."""
        if self._fexec:
            return self.lib.dm_fexec_compute_stream(self._fexec)
        return self.lib.dm_exec_compute_stream(self._exec)

    def enqueue_wait_ack(self) -> None:
        """Stream-ordered fence: the compute stream does not proceed until the PS has applied every push made so
        far (mailbox mode). Used to close a device-timed region on the PS-side apply of its last step."""
        if self.cfg.backend != "cuda":
            return
        if self._exec:
            N.check(self.lib.dm_exec_join(self._exec), "join lanes")   # lane 0 now follows every in-flight step
        if self.cfg.push_mode == "mailbox" and self.inbox_order:
            N.check(self.lib.dm_launch_wait_ack(self.seg.addr("inbox"), len(self.inbox_order), self._seq_word_ptr(),
                                                self.compute_stream), "wait_ack")

    def fork_lanes(self) -> None:
        """Every lane waits for what is enqueued on lane 0 (e.g. a timing event) before running further steps."""
        if self.cfg.backend == "cuda" and self._exec:
            N.check(self.lib.dm_exec_fork(self._exec), "fork lanes")

    def kernel_launches(self) -> int:
        if self._fexec:
            return int(self.lib.dm_fexec_launches(self._fexec))
        return int(self.lib.dm_exec_kernel_launches(self._exec)) if self._exec else 0

    # ------------------------------------------------------------------------------------------
    # CPU backend step (same protocol, torch math)
    # ------------------------------------------------------------------------------------------
    def _cpu_views(self):
        if getattr(self, "_views", None) is None:
            self._views = []
            for k, seg in enumerate(self.ps_segs):
                d = self.ps_desc[k]
                arena, ni = d["arena_elems"], max(d.get("n_flags", d["n_items"]), 1)
                w, ns = self.task_index, self.cfg.nslots
                self._views.append({
                    "params": seg.tensor("params", torch.float32),
                    "mailbox": seg.tensor("mailbox", torch.float32).view(self.cluster.num_workers, ns, arena)[w],
                    "flags_addr": seg.addr("flags", w * ns * ni * 4),
                    "ni": ni,
                })
            self._inbox_addr = self.seg.addr("inbox")
        return self._views

    def _cpu_step(self, x: torch.Tensor, y: torch.Tensor) -> StepOutput:
        views = self._cpu_views()
        lay = self.layout
        # pull (X3): snapshot of the live shard memory; concurrent applies may tear it (Hogwild, like the reference)
        params = {}
        for name, vl in lay.by_name.items():
            if len({(pc.ps, pc.offset) for pc in vl.pieces}) == 1:
                flat = views[vl.ps]["params"][vl.offset: vl.offset + vl.span]
                params[name] = self._unpack(vl, flat)
            else:   # column-split variable: every owning shard holds the live values of its own columns
                full = torch.empty(vl.rows, vl.cols)
                for pc in vl.pieces:
                    if pc.c1 > pc.c0:
                        src = self._unpack(vl, views[pc.ps]["params"][pc.offset: pc.offset + vl.span])
                        full[:, pc.c0:pc.c1] = src[:, pc.c0:pc.c1]
                params[name] = full
        loss, grads, logits = mlp.manual_loss_and_grads(self.spec, params, x.float(), y.float())
        correct = mlp.accuracy_count(logits, y)
        self._seq_host += 1
        seq, ns = self._seq_host, self.cfg.nslots
        slot = seq % ns
        if seq > ns:  # flow control: wait until push (seq - nslots) has been applied everywhere
            for k, i in self.inbox_index.items():
                if self.lib.dm_wait_ge_u32(self._inbox_addr + 8 * i, seq - ns, 120.0) != 0:
                    raise TimeoutError(f"ps {k} did not acknowledge push {seq - ns}")
        # push (X4): gradients into our mailbox slot, then publish every item's flag
        for name, vl in lay.by_name.items():
            packed = self._pack(vl, grads[name])
            for k, off in dict.fromkeys((pc.ps, pc.offset) for pc in vl.pieces):
                views[k]["mailbox"][slot, off: off + vl.span] = packed
        for k in self.inbox_order:
            v = views[k]
            for flag in range(lay.shards[k].n_flags):
                self.lib.dm_store_release_u32(v["flags_addr"] + 4 * (slot * v["ni"] + flag), seq)
        if self.inbox_order and self.cfg.strict_steps:
            # --strict_steps (reference order inside one worker, DS:110-113): the step returns — and the next pull
            # happens — only after every shard has applied this push
            for k, i in self.inbox_index.items():
                if self.lib.dm_wait_ge_u32(self._inbox_addr + 8 * i, seq, 120.0) != 0:
                    raise TimeoutError(f"ps {k} did not acknowledge push {seq}")
        if self.inbox_order:
            ack = self.lib.dm_load_acquire_u32(self._inbox_addr)
            gstep = self.lib.dm_load_acquire_u32(self._inbox_addr + 4) + (seq - ack)
        else:
            gstep = seq
        return StepOutput(float(loss), int(gstep), int(correct), seq)

    # ------------------------------------------------------------------------------------------
    # evaluation (forward only, accuracy kernel / torch on cpu)
    # ------------------------------------------------------------------------------------------
    @nvtx_annotate("dm.worker.evaluate")
    def evaluate(self, images: torch.Tensor, labels: torch.Tensor) -> Tuple[float, float]:
        """(mean loss, accuracy) of the current PS variables on a host dataset; GPU path uses the hand-written
        accuracy reduction kernel (SURVEY K12) on torch-computed logits of the pulled variables."""
        if self.cfg.backend == "cuda" and self.engine == "fused":
            # Evaluation is not part of a training step: logits of the pulled variables are computed with torch on the
            # host (no torch CUDA kernel is launched — a lazily loaded kernel could deadlock against a resident
            # persistent ps kernel of an in-process cluster), the correct-prediction count with the hand-written,
            # pre-loaded accuracy reduction (SURVEY K12) on pre-allocated device buffers.
            self.drain()
            params = self.read_variables()
            logits, _ = mlp.forward_logits(self.spec, params, images.float())
            logits = logits.float().contiguous()
            labels_f = labels.float().contiguous()
            loss = float(mlp.loss_from_logits(self.spec, logits, labels_f))
            stream = self.compute_stream
            Cn, cap = self.spec.num_classes, self._ev_rows
            correct = 0
            for r0 in range(0, logits.shape[0], cap):
                n = min(cap, logits.shape[0] - r0)
                self._ev_pin[:n].copy_(logits[r0:r0 + n])
                self._ev_pin[cap:cap + n].copy_(labels_f[r0:r0 + n])
                self._ev_cnt_pin.zero_()
                N.check(self.lib.dm_memcpy_async(self._ev_dev.data_ptr(), self._ev_pin.data_ptr(), n * Cn * 4, stream))
                N.check(self.lib.dm_memcpy_async(self._ev_dev.data_ptr() + cap * Cn * 4,
                                                 self._ev_pin.data_ptr() + cap * Cn * 4, n * Cn * 4, stream))
                N.check(self.lib.dm_memcpy_async(self._ev_cnt.data_ptr(), self._ev_cnt_pin.data_ptr(), 4, stream))
                N.check(self.lib.dm_launch_accuracy(self._ev_dev.data_ptr(), self._ev_dev.data_ptr() + cap * Cn * 4, n, Cn,
                                                    self._ev_cnt.data_ptr(), stream), "accuracy kernel")
                N.check(self.lib.dm_memcpy_async(self._ev_cnt_pin.data_ptr(), self._ev_cnt.data_ptr(), 4, stream))
                N.check(self.lib.dm_stream_sync(stream))
                correct += int(self._ev_cnt_pin.item())
            return loss, correct / max(1, images.shape[0])
        if self.cfg.backend == "cuda":
            # forward tcgen05 GEMMs (weights pulled from the PS shards) + the head kernel in eval mode; whole
            # batches only (the step kernels are specialised for this worker's batch size).
            self.drain()
            stream = self.compute_stream
            n_chunks = images.shape[0] // self.batch
            if n_chunks == 0:
                raise ValueError(f"evaluate needs at least one full batch of {self.batch} samples")
            xs = torch.zeros(self.B_pad, self.ld_in, dtype=self.tdtype).pin_memory()
            ys = torch.zeros(self.B_pad, self.spec.num_classes, dtype=torch.float32).pin_memory()
            res = torch.zeros(4, dtype=torch.int32).pin_memory()
            loss_sum, correct = 0.0, 0
            for c in range(n_chunks):
                sl = slice(c * self.batch, (c + 1) * self.batch)
                xs[: self.batch, : images.shape[1]].copy_(images[sl])
                ys[: self.batch].copy_(labels[sl])
                N.check(self.lib.dm_memcpy_async(self._eval_x.data_ptr(), xs.data_ptr(), xs.numel() * xs.element_size(), stream))
                N.check(self.lib.dm_memcpy_async(self._eval_y.data_ptr(), ys.data_ptr(), ys.numel() * 4, stream))
                for p in self._eval_plans:
                    p.launch(stream)
                N.check(self.lib.dm_memcpy_async(res.data_ptr(), self._eval_res.data_ptr(), 16, stream))
                N.check(self.lib.dm_stream_sync(stream))
                loss_sum += float(res[:1].view(torch.float32).item())
                correct += int(res[2].item())
            return loss_sum / n_chunks, correct / (n_chunks * self.batch)
        params = self.read_variables()
        logits, _ = mlp.forward_logits(self.spec, params, images.float())
        correct = mlp.accuracy_count(logits, labels)
        loss = float(mlp.loss_from_logits(self.spec, logits, labels.float()))
        return loss, correct / max(1, images.shape[0])

    # ------------------------------------------------------------------------------------------
    # teardown
    # ------------------------------------------------------------------------------------------
    def finish(self) -> None:
        """Leave the session: tell every PS shard how many pushes we made so its serve kernel can retire us."""
        if not self._connected or getattr(self, "_finished", False):
            return
        self._finished = True
        w = self.task_index
        if self.cfg.push_mode == "mailbox":
            # every shard hears it, also one that owns no variable (its serve loop only waits for this word)
            if self.cfg.backend == "cuda" and (self._exec or self._fexec):
                self.drain()
                stream = self.compute_stream
                for k in range(self.cluster.num_ps):
                    N.check(self.lib.dm_launch_worker_done(self.ps_segs[k].addr("ctrl", 4 * (CTRL_WORKER_DONE + w)),
                                                           self._seq_word_ptr(), stream))
                N.check(self.lib.dm_stream_sync(stream))
                self._serve_local()
            elif self.cfg.backend == "cpu":
                for k in range(self.cluster.num_ps):
                    self.lib.dm_store_release_u32(self.ps_segs[k].addr("ctrl", 4 * (CTRL_WORKER_DONE + w)),
                                                  self._seq_host + 1)
        self.rdv.put(f"session/done/{w}", 1)
        self.rdv.add("session/workers_done", 1)

    def close(self) -> None:
        if self._closed:
            return
        self._closed = True
        if getattr(self, "_hb_thread", None) is not None:
            self._hb_stop.set()
        self.finish()
        if self._exec:
            self.lib.dm_exec_destroy(self._exec)
            self._exec = None
        if self._fexec:
            self.lib.dm_fexec_destroy(self._fexec)
            self._fexec = None
        self._views = None
        for seg in self.ps_segs:
            seg.close()
        if self.seg is not None:
            self.seg.close()


class NativeLoader:
    """Host dataset + native `next_batch` loader (TF DataSet.next_batch semantics, csrc/loader.h).

    Fused engine on cuda: the loader keeps an *epoch feed* — like TF's DataSet it holds the rows of an epoch physically
    in shuffled order (two pinned buffers: current and next epoch), so a batch is a contiguous slice of pinned memory
    that the executor DMAs to the GPU without touching it; the next epoch's buffer is filled by the executor's helper
    threads while the current one is consumed (csrc/fused_exec.cu). ``epoch_feed=False`` (or ``DM_EPOCH_FEED=0``)
    keeps the row-gather path for every batch."""

    def __init__(self, worker: Worker, images: torch.Tensor, labels: torch.Tensor, seed: int = 0, shuffle: bool = True,
                 epoch_feed: Optional[bool] = None):
        self.worker = worker
        self.images = images.to(worker.tdtype).contiguous()
        self.labels = labels.to(torch.float32).contiguous()
        n, pix = self.images.shape
        es = self.images.element_size()
        ncls = self.labels.shape[1]
        if epoch_feed is None:
            epoch_feed = os.environ.get("DM_EPOCH_FEED", "1") != "0"
        want_feed = (epoch_feed and worker.cfg.backend == "cuda" and worker.engine == "fused"
                     and worker.batch == N.FUSED_ROWS_PER_SLOT and worker.ld_in == pix and n >= 1024)
        if worker.cfg.backend == "cuda" and not want_feed:
            self.images = self.images.pin_memory()
            self.labels = self.labels.pin_memory()
        self.handle = worker.lib.dm_loader_create(
            self.images.data_ptr(), self.labels.data_ptr(), n, pix * es, ncls * 4,
            worker.ld_in * es, ncls * 4, worker.batch, seed, int(shuffle))
        # destroyed when the object is collected or at interpreter exit — in both cases *before* the tensors above are
        # released (a weakref finalizer runs ahead of the instance's own teardown)
        self._finalizer = weakref.finalize(self, worker.lib.dm_loader_destroy, self.handle)
        self._feed_bufs = None
        if want_feed:
            # allocated here, where the dataset used to be pinned: before an in-process ps kernel becomes resident
            try:
                bufs = [torch.empty((n, pix), dtype=worker.tdtype, pin_memory=True) for _ in range(2)]
                bufs += [torch.empty((n, ncls), dtype=torch.float32, pin_memory=True) for _ in range(2)]
            except RuntimeError as e:   # no room for two pinned copies of the dataset: keep the row-gather path
                print(f"[worker {worker.task_index}] epoch feed disabled (pinned allocation failed: {e})", flush=True)
                bufs = None
            helpers = max(1, min(8, usable_cores() // 2))
            if bufs is not None and worker.lib.dm_loader_enable_feed(
                    self.handle, bufs[0].data_ptr(), bufs[2].data_ptr(), bufs[1].data_ptr(), bufs[3].data_ptr(),
                    helpers) == 1:
                self._feed_bufs = bufs   # kept alive with the loader
        self._xbuf = torch.zeros(worker.batch, worker.ld_in, dtype=worker.tdtype)
        self._ybuf = torch.zeros(worker.batch, self.labels.shape[1], dtype=torch.float32)

    @property
    def epoch_feed(self) -> bool:
        return self._feed_bufs is not None

    def next_batch(self) -> Tuple[torch.Tensor, torch.Tensor]:
        self.worker.lib.dm_loader_next(self.handle, self._xbuf.data_ptr(), self._ybuf.data_ptr())
        return self._xbuf[:, : self.images.shape[1]].clone(), self._ybuf.clone()

    @property
    def epochs(self) -> int:
        return int(self.worker.lib.dm_loader_epochs(self.handle))

    def close(self) -> None:
        """Destroy the native loader (waits for an epoch fill that is still running on the executor's helper threads:
        they read the dataset and write the feed buffers this object owns)."""
        self._finalizer()
        self.handle = None
