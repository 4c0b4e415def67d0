"""Data-parallel SAE training over NVLink peer memory (csrc/p2p.cu) -- host side.

``P2PGroup`` allocates peer-visible buffers through the library (cudaMalloc + CUDA IPC handle), swaps the 64-byte
handles between the ranks ONCE (``torch.distributed.all_gather_object`` -- plumbing, not the data path) and opens every
peer's buffers.  ``SaeDPEngine`` is ``SaeStepEngine`` with its parameters, gradients and a few small vectors living in
those buffers and the optimizer step replaced by reduce-scatter (peer loads) -> clip/project/Adam on the owned row
slice -> all-gather (peer stores).  Single-GPU semantics are preserved: the loss is the mean over the GLOBAL batch
(column mean of x, 1/(tokens*d) factor), the clip norm is that of the summed gradient, dead-feature counters are summed.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Callable, Dict, List, Optional

import torch

from . import _lib as L
from .ops import _stream
from .sae_engine import PbSaeEncode, PbSaeStep, SaeStepEngine, ops_cast_f32

vp, i32, i64, f32, u32, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint32, C.c_uint64
MAX_RANKS = 8
_TABLES = ("gW_dec", "gW_encT", "gb_enc", "gb_dec", "fired", "xsum", "W_dec", "W_encT", "W_encT_lo", "b_enc", "norm_parts", "flags")


class PbP2PStep(C.Structure):
    _fields_ = (
        [(n, i32) for n in ("rank", "world", "d", "F", "step", "global_rows")]
        + [(n, f32) for n in ("lr", "beta1", "beta2", "adam_eps", "max_grad_norm")]
        + [(n, vp * MAX_RANKS) for n in _TABLES]
        + [(n, vp) for n in ("gb_enc_red", "gb_dec_red", "fired_red", "part_accum", "b_dec", "scalars",
                             "m_dec", "v_dec", "m_enc", "v_enc", "m_be", "v_be", "m_bd", "v_bd", "since_fired", "act_freq")]
        + [(n, vp) for n in ("mc_gW_dec", "mc_gW_encT", "mc_W_dec", "mc_W_encT", "mc_b_enc")]     # NVSwitch multicast views (or NULL)
        + [("defer_dec", i32)]
    )


L.ABI_STRUCTS.extend([None, PbP2PStep, PbSaeEncode])   # 7 = device-side scalars struct (no ctypes twin), 8 = PbP2PStep, 9 = PbSaeEncode
L.register_signatures({
    "pb_p2p_alloc": (i32, [i64, C.POINTER(vp), C.c_char_p]),
    "pb_p2p_open": (i32, [C.c_char_p, C.POINTER(vp)]),
    "pb_p2p_close": (i32, [vp]),
    "pb_p2p_free": (i32, [vp]),
    "pb_p2p_barrier": (i32, [C.POINTER(PbP2PStep), u32, vp]),
    "pb_p2p_sum_xsum": (i32, [C.POINTER(PbP2PStep), vp, vp]),
    "pb_p2p_reduce_scatter": (i32, [C.POINTER(PbP2PStep), vp]),
    "pb_p2p_adam_allgather": (i32, [C.POINTER(PbP2PStep), vp]),
    "pb_p2p_push_dec": (i32, [C.POINTER(PbP2PStep), vp]),
    "pb_mc_supported": (i32, [C.POINTER(i32)]),
    "pb_mc_round_size": (i32, [i32, i64, C.POINTER(i64)]),
    "pb_mc_create": (i32, [i32, i64, C.POINTER(u64), C.POINTER(i32)]),
    "pb_mc_import": (i32, [i32, C.POINTER(u64)]),
    "pb_mc_add_device": (i32, [u64]),
    "pb_mc_bind_alloc": (i32, [u64, i64, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]),
})


def shard_bounds(F: int, rank: int, world: int):
    """Feature rows owned by ``rank``: contiguous, equal slices (F must divide evenly -- d_sae is d_in * expansion)."""
    if F % world:
        raise ValueError(f"d_sae={F} is not divisible by world size {world}")
    per = F // world
    return rank * per, (rank + 1) * per


class _RawCuda:
    """Minimal ``__cuda_array_interface__`` carrier so torch can view library-owned device memory without copying."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 3, "strides": None}


_TYPESTR = {torch.float32: "<f4", torch.int32: "<i4", torch.uint8: "|u1"}


class P2PGroup:
    def __init__(self, rank: int, world: int, device: torch.device, exchange: Optional[Callable[[dict], List[dict]]] = None):
        if not 1 <= world <= MAX_RANKS:
            raise ValueError(f"world size {world} outside 1..{MAX_RANKS}")
        self.rank, self.world, self.device = rank, world, device
        self._exchange = exchange or self._exchange_dist
        self.local: Dict[str, torch.Tensor] = {}
        self._ptr: Dict[str, int] = {}
        self._handle: Dict[str, bytes] = {}
        self.peer_ptr: Dict[str, List[int]] = {}
        self.epoch = 0

    @staticmethod
    def _exchange_dist(mine: dict) -> List[dict]:
        import torch.distributed as dist
        out = [None] * dist.get_world_size()
        dist.all_gather_object(out, mine)
        return out

    def alloc(self, name: str, shape, dtype=torch.float32) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= s
        nbytes = max(n, 1) * torch.empty((), dtype=dtype).element_size()
        ptr = vp()
        handle = C.create_string_buffer(64)
        L.check(L.get_lib().pb_p2p_alloc(nbytes, C.byref(ptr), handle), "pb_p2p_alloc")
        t = torch.as_tensor(_RawCuda(ptr.value, shape, _TYPESTR[dtype]), device=self.device)
        self.local[name], self._ptr[name], self._handle[name] = t, ptr.value, handle.raw
        return t

    # ------------------------------------------------------------------ NVSwitch multicast pool (csrc/mc.cu)
    def try_multicast_pool(self, nbytes: int):
        """COLLECTIVE.  One multicast object + one bound physical allocation per rank, ``nbytes`` (rounded up) each.  Returns
        ``(own_ptr, multicast_ptr, rounded_bytes)`` or ``None`` when the fabric / driver does not support it or any rank failed
        (every rank then takes the peer load / store path).  The multicast handle travels as a POSIX file descriptor over a
        Unix-domain socket (SCM_RIGHTS); torch.distributed only carries the socket path and the go / no-go votes."""
        import os
        import socket
        import tempfile
        import torch.distributed as dist
        lib = L.get_lib()
        # Opt-in (PRISMA_P2P_MULTICAST=1).  Measured on 2 and 8 B200s (profiles/r02_dp_notes.md): multimem.ld_reduce makes every GPU
        # send its WHOLE gradient through its link once (the switch pulls each rank's copy of every slice, the requester's own
        # included), the peer-load reduce-scatter sends (N-1)/N of it; ingress shrinks to 1/N but the links are full duplex, so the
        # exchange time is the same at 8 ranks (1.151 vs 1.146 ms/step) and worse at 2 (1.20 vs 1.01).
        if os.environ.get("PRISMA_P2P_MULTICAST", "0") != "1" or not (dist.is_available() and dist.is_initialized()):
            self.multicast_note = "NVSwitch multicast available with PRISMA_P2P_MULTICAST=1; not faster than peer loads / stores here"
            return None

        def all_ok(flag: bool) -> bool:
            t = torch.tensor([1 if flag else 0], device=self.device, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return bool(t.item())

        sup = i32(0)
        lib.pb_mc_supported(C.byref(sup))
        if not all_ok(bool(sup.value)):
            self.multicast_note = "multicast not supported on this device / fabric"
            return None
        rounded = i64(0)
        ok = lib.pb_mc_round_size(self.world, int(nbytes), C.byref(rounded)) == L.PB_OK
        if not all_ok(ok):
            self.multicast_note = "multicast granularity query failed: " + L.last_error()
            return None
        handle, fd, sock_path, srv = u64(0), i32(-1), [None], None
        if self.rank == 0:
            ok = lib.pb_mc_create(self.world, rounded.value, C.byref(handle), C.byref(fd)) == L.PB_OK
            if ok:
                sock_path[0] = os.path.join(tempfile.gettempdir(), f"prisma_mc_{os.getpid()}_{id(self) & 0xffff:x}.sock")
                srv = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
                if os.path.exists(sock_path[0]):
                    os.unlink(sock_path[0])
                srv.bind(sock_path[0])
                srv.listen(self.world)
        if not all_ok(ok):
            self.multicast_note = "cuMulticastCreate failed: " + L.last_error()
            return None
        dist.broadcast_object_list(sock_path, src=0)
        try:
            if self.rank == 0:
                for _ in range(self.world - 1):
                    conn, _addr = srv.accept()
                    socket.send_fds(conn, [b"mc"], [fd.value])
                    conn.close()
                srv.close()
                os.unlink(sock_path[0])
            else:
                cli = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
                cli.connect(sock_path[0])
                _msg, fds, _flags, _addr = socket.recv_fds(cli, 16, 1)
                cli.close()
                ok = len(fds) == 1 and lib.pb_mc_import(fds[0], C.byref(handle)) == L.PB_OK
        except OSError as e:       # noqa: PERF203
            ok = False
            self.multicast_note = f"fd exchange failed: {e}"
        if not all_ok(ok):
            self.multicast_note = getattr(self, "multicast_note", "") or ("multicast import failed: " + L.last_error())
            return None
        ok = lib.pb_mc_add_device(handle.value) == L.PB_OK
        if not all_ok(ok):                       # doubles as the barrier "every device joined" that must precede the binds
            self.multicast_note = "cuMulticastAddDevice failed: " + L.last_error()
            return None
        own, mc, mem = vp(), vp(), u64(0)
        ok = lib.pb_mc_bind_alloc(handle.value, rounded.value, C.byref(own), C.byref(mc), C.byref(mem)) == L.PB_OK
        if not all_ok(ok):                       # barrier: every rank has bound before anybody touches the multicast view
            self.multicast_note = "multicast bind / map failed: " + L.last_error()
            return None
        self.multicast_note = f"NVSwitch multicast pool, {rounded.value >> 20} MiB per rank"
        return own.value, mc.value, rounded.value

    def connect(self) -> None:
        """Swap IPC handles and open every peer's buffers (collective: call on all ranks after all ``alloc`` calls)."""
        everyone = self._exchange(dict(self._handle))
        for name in self._handle:
            ptrs = []
            for r in range(self.world):
                if r == self.rank:
                    ptrs.append(self._ptr[name])
                    continue
                peer = vp()
                L.check(L.get_lib().pb_p2p_open(everyone[r][name], C.byref(peer)), f"pb_p2p_open({name}, rank {r})")
                ptrs.append(peer.value)
            self.peer_ptr[name] = ptrs

    def fill_tables(self, s: PbP2PStep) -> None:
        s.rank, s.world = self.rank, self.world
        for name in _TABLES:
            if name not in self.peer_ptr:              # optional table (W_encT_lo): stays NULL
                continue
            arr = getattr(s, name)
            for r, p in enumerate(self.peer_ptr[name]):
                arr[r] = p

    def barrier(self, s: PbP2PStep) -> None:
        self.epoch += 1
        L.check(L.get_lib().pb_p2p_barrier(C.byref(s), self.epoch, _stream()), "pb_p2p_barrier")

    def barrier2(self, s: PbP2PStep, stream: int) -> None:
        """Barrier of the side stream: its own flag words ("flags2") and epoch counter, so it can interleave with ``barrier``."""
        self.epoch2 = getattr(self, "epoch2", 0) + 1
        flags = s.flags
        saved = [flags[r] for r in range(MAX_RANKS)]
        for r, p in enumerate(self.peer_ptr["flags2"]):
            flags[r] = p
        try:
            L.check(L.get_lib().pb_p2p_barrier(C.byref(s), self.epoch2, stream), "pb_p2p_barrier(side)")
        finally:
            for r in range(MAX_RANKS):
                flags[r] = saved[r]


class SaeDPEngine(SaeStepEngine):
    """``SaeStepEngine`` whose optimizer step is the NVLink reduce-scatter / sharded Adam / all-gather of csrc/p2p.cu."""
    is_data_parallel = True

    def __init__(self, group: P2PGroup, W_encT: torch.Tensor, W_dec: torch.Tensor, b_enc: torch.Tensor, b_dec: torch.Tensor, k: int, **kw):
        self.group = group
        F, d = W_dec.shape
        shard_bounds(F, group.rank, group.world)
        g = group
        # parameters + gradient matrices: one NVSwitch multicast pool when the fabric offers it (multimem.ld_reduce / multimem.st in
        # p2p.cu), else IPC-shared cudaMalloc buffers (peer loads / stores).  The dense 3xTF32 encoder needs its residual plane
        # all-gathered too and stays on the peer path.
        big = ("W_encT", "W_dec", "gW_dec", "gW_encT")
        self.mc = None
        pool = None
        fused_geometry = d % 4 == 0 and d >= 32 and F % 128 == 0 and k <= 48 and F <= 131072      # SaeStepEngine's fused-encoder rule
        if fused_geometry and kw.get("encoder", "auto") != "dense" and kw.get("gemm_impl", L.GEMM_AUTO) == L.GEMM_AUTO:
            rowb = -(-F // 64) * 256                                   # b_enc, padded to 256 bytes
            pool = g.try_multicast_pool(4 * F * d * 4 + rowb)
        if pool is not None:
            own, mcp, _size = pool
            offs = {name: i * F * d * 4 for i, name in enumerate(big)}
            offs["b_enc"] = 4 * F * d * 4
            shared = {}
            for name in big + ("b_enc",):
                shape = (F, d) if name != "b_enc" else (F,)
                t = torch.as_tensor(_RawCuda(own + offs[name], shape, "<f4"), device=g.device)
                g.local[name], g.peer_ptr[name] = t, [own + offs[name] if r == g.rank else 0 for r in range(g.world)]
                shared[name] = t
            self.mc = {name: mcp + offs[name] for name in offs}
        else:
            shared = {"W_encT": g.alloc("W_encT", (F, d)), "W_dec": g.alloc("W_dec", (F, d)), "b_enc": g.alloc("b_enc", (F,))}
            for name in ("gW_dec", "gW_encT"):
                g.alloc(name, (F, d))
        shared["W_encT"].copy_(W_encT)
        shared["W_dec"].copy_(W_dec)
        shared["b_enc"].copy_(b_enc)
        for name, shape in (("gb_enc", (F,)), ("gb_dec", (d,)), ("fired", (F,)), ("xsum", (d,)), ("norm_parts", (MAX_RANKS,))):
            g.alloc(name, shape)
        g.alloc("flags", (MAX_RANKS,), dtype=torch.int32)
        g.alloc("flags2", (MAX_RANKS,), dtype=torch.int32)        # barrier of the side stream that finishes the W_dec all-gather
        super().__init__(shared["W_encT"], shared["W_dec"], shared["b_enc"], b_dec.clone().contiguous(), k, **kw)
        # re-point the buffers peers must reach at the shared allocations
        if self.W_encT_lo is not None:                 # dense 3xTF32 encoder: the residual plane is all-gathered with the parameters
            self.W_encT_lo = g.alloc("W_encT_lo", (F, d))
            self.refresh_lo()
        self.gW_dec, self.gW_encT, self.gb_enc, self.gb_dec = g.local["gW_dec"], g.local["gW_encT"], g.local["gb_enc"], g.local["gb_dec"]
        self.fired = g.local["fired"]
        self.xsum_local = g.local["xsum"]
        dev = W_dec.device
        self.gb_enc_red, self.gb_dec_red, self.fired_red = torch.zeros(F, device=dev), torch.zeros(d, device=dev), torch.zeros(F, device=dev)
        self.part_accum = torch.zeros(4, device=dev)        # [0]: gradient-norm partial of the owned slice
        import os
        # PRISMA_P2P_OVERLAP=1: the W_dec half of the all-gather runs on a side stream under the next step's prep / encoder GEMM /
        # select (it is first read by the next decode).  OFF by default: measured no gain at 8 ranks and a loss at 2 (run 17's trace:
        # the SM-driven push kernel slows the concurrent candidate GEMM by as much as the Adam kernel gets shorter); a copy-engine
        # push would not share SMs with the GEMM -- not built.
        self.overlap_dec = os.environ.get("PRISMA_P2P_OVERLAP", "0") == "1" and g.world > 1
        self._side = torch.cuda.Stream(device=dev) if self.overlap_dec else None
        self._trace = [] if os.environ.get("PRISMA_P2P_TRACE", "0") == "1" else None      # per-step CUDA-event marks (trace_report)
        self._trace_step = []
        self._ev_adam = torch.cuda.Event() if self.overlap_dec else None
        self._ev_dec = None                                   # recorded on the side stream once every peer's W_dec rows have landed
        g.connect()
        torch.cuda.synchronize()

    def _p2p_desc(self, rows: int, lr: float, since_fired, act_freq) -> PbP2PStep:
        s = PbP2PStep()
        self.group.fill_tables(s)
        s.d, s.F, s.step, s.global_rows = self.d, self.F, self.step_count, rows * self.group.world
        s.lr, s.beta1, s.beta2, s.adam_eps, s.max_grad_norm = lr, self.betas[0], self.betas[1], self.adam_eps, self.max_grad_norm
        p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        s.gb_enc_red, s.gb_dec_red, s.fired_red, s.part_accum = p(self.gb_enc_red), p(self.gb_dec_red), p(self.fired_red), p(self.part_accum)
        s.b_dec, s.scalars = p(self.b_dec), p(self.scalars)
        s.m_dec, s.v_dec, s.m_enc, s.v_enc = p(self.m_dec), p(self.v_dec), p(self.m_enc), p(self.v_enc)
        s.m_be, s.v_be, s.m_bd, s.v_bd = p(self.m_be), p(self.v_be), p(self.m_bd), p(self.v_bd)
        s.since_fired, s.act_freq = p(since_fired), p(act_freq)
        if self.mc is not None:
            s.mc_gW_dec, s.mc_gW_encT = self.mc["gW_dec"], self.mc["gW_encT"]
            s.mc_W_dec, s.mc_W_encT, s.mc_b_enc = self.mc["W_dec"], self.mc["W_encT"], self.mc["b_enc"]
        return s

    def wait_parameters(self) -> None:
        """Make the current stream wait for the deferred W_dec all-gather of the last step (call before reading W_dec outside
        ``train_step``: forward(), state_dict(), checkpoints)."""
        if self._ev_dec is not None:
            torch.cuda.current_stream().wait_event(self._ev_dec)
            self._ev_dec = None

    @torch.no_grad()
    def forward(self, x: torch.Tensor, want_out: bool = True):
        self.wait_parameters()
        return super().forward(x, want_out)

    def describe_exchange(self) -> str:
        n = self.group.world
        if self.mc is not None:
            return (f"NVSwitch multicast: reduce-scatter by multimem.ld_reduce (summed in the switch), all-gather by multimem.st; "
                    f"{int(2 * 8 * self.d * self.F / n / 1e6)} MB over NVLink per GPU per step")
        return (f"peer loads / stores over NVLink: {int((n - 1) / n * (2 * self.d * self.F * 4 * 2) / 1e6)} MB per GPU per step"
                + (f" ({getattr(self.group, 'multicast_note', '')})" if getattr(self.group, "multicast_note", "") else ""))

    # ------------------------------------------------------------------ PRISMA_P2P_TRACE=1: CUDA events at the phase boundaries of every step
    def _mark(self, name: str, stream=None) -> None:
        if self._trace is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(stream if stream is not None else torch.cuda.current_stream())
        self._trace_step.append((name, ev))

    def trace_report(self, skip: int = 5) -> dict:
        """Mean milliseconds between consecutive marks of a step (main stream) and, for marks on the side stream, since the step's
        first mark.  Synchronises."""
        if not self._trace:
            return {}
        torch.cuda.synchronize()
        steps = self._trace[skip:] or self._trace
        out, n = {}, len(steps)
        for marks in steps:
            t0, prev = marks[0][1], marks[0][1]
            for name, ev in marks[1:]:
                if name.startswith("side:"):
                    out[name + " (since step start)"] = out.get(name + " (since step start)", 0.0) + t0.elapsed_time(ev) / n
                else:
                    out[name] = out.get(name, 0.0) + prev.elapsed_time(ev) / n
                    prev = ev
            out["step total"] = out.get("step total", 0.0) + t0.elapsed_time(prev) / n
        return {k: round(v, 4) for k, v in out.items()}

    @torch.no_grad()
    def train_step(self, x: torch.Tensor, lr: float, since_fired=None, act_freq=None, want_out: bool = False) -> torch.Tensor:
        lib, st, g = L.get_lib(), _stream(), self.group
        x = ops_cast_f32(x)
        rows = x.shape[0]
        if getattr(self, "_dp_rows", rows) != rows:
            raise L.PrismaB200Error(f"SaeDPEngine: every step (and every rank) must bring the same number of rows (had {self._dp_rows}, got {rows}); "
                                    "drop or pad short batches before the data-parallel step")
        self._dp_rows = rows
        if self._trace is not None:
            self._trace_step = []
            self._trace.append(self._trace_step)
        self._mark("start")
        # prep writes THIS rank's column sums of x into the shared xsum; decode needs the GLOBAL sums
        self._ensure_rows(rows)
        self.step_count += 1
        s = self._desc(x, training=True, lr=float(lr), since_fired=since_fired, act_freq=act_freq, want_out=want_out)
        s.global_rows, s.dist, s.pre_zeroed = rows * g.world, 1, 1
        L.check(lib.pb_sae_step_reset(C.byref(s), self.fb_count.data_ptr(), st), "pb_sae_step_reset")     # every accumulator of the step, one launch
        xsum_global, self.xsum = self.xsum, self.xsum_local
        self.encode_topk(x, pre_zeroed=True)
        self.xsum = xsum_global
        self._mark("reset + prep + encode + topk")
        ps = self._p2p_desc(rows, float(lr), since_fired, act_freq)
        g.barrier(ps)
        L.check(lib.pb_p2p_sum_xsum(C.byref(ps), self.xsum.data_ptr(), st), "pb_p2p_sum_xsum")
        self._mark("barrier + xsum")
        if self._ev_dec is not None:                    # the previous step's W_dec rows from every peer (side stream) must have landed
            torch.cuda.current_stream().wait_event(self._ev_dec)
            self._ev_dec = None
            self._mark("wait for the deferred W_dec rows")
        L.check(lib.pb_sae_decode(C.byref(s), st), "pb_sae_decode")
        self._mark("decode")
        L.check(lib.pb_sae_backward(C.byref(s), st), "pb_sae_backward")
        self._mark("backward")
        g.barrier(ps)                                   # every rank's local gradients are complete
        self._mark("barrier (gradients complete)")
        L.check(lib.pb_p2p_reduce_scatter(C.byref(ps), st), "pb_p2p_reduce_scatter")
        self._mark("reduce-scatter")
        g.barrier(ps)                                   # norm partials published; all peer reads of this step are done
        self._mark("barrier (norm parts)")
        ps.defer_dec = 1 if self.overlap_dec else 0
        L.check(lib.pb_p2p_adam_allgather(C.byref(ps), st), "pb_p2p_adam_allgather")
        self._mark("sharded Adam + all-gather")
        g.barrier(ps)                                   # every rank holds the updated encoder (and, without overlap, decoder) parameters
        self._mark("barrier (parameters)")
        if self.overlap_dec:
            # W_dec rows -> peers on the side stream with its own flag set, started AFTER the encoder all-gather has completed everywhere:
            # started together with it (run 13) the two pushes shared the egress links and the barrier above waited for both -- no gain.
            # From here the traffic runs under the next step's prep / candidate GEMM / select and is awaited at its decode.
            self._ev_adam.record(torch.cuda.current_stream())
            self._side.wait_event(self._ev_adam)
            side = self._side.cuda_stream
            self._mark("side: push start", self._side)
            L.check(lib.pb_p2p_push_dec(C.byref(ps), side), "pb_p2p_push_dec")
            self._mark("side: push done", self._side)
            g.barrier2(ps, side)
            self._mark("side: barrier2 done", self._side)
            self._ev_dec = torch.cuda.Event()
            self._ev_dec.record(self._side)
        if self.encoder == "fused":
            # the next step's candidate GEMM reads the fp16 shadow and the encoder-row norm maxima: every rank rebuilds both from its
            # full, freshly all-gathered W_encT (one local pass; the shadow rows are not pushed over NVLink)
            self.refresh_lo()
        self._mark("fp16 shadow refresh")
        return self.scalars

    # ------------------------------------------------------------------ instrumentation: COLLECTIVE (every rank must call it)
    def _prepare_timed_step(self, s: PbSaeStep, x: torch.Tensor) -> None:
        s.global_rows, s.dist = x.shape[0] * self.group.world, 1

    def _optimizer_stages(self, s: PbSaeStep, x: torch.Tensor, lr: float, since_fired, act_freq):
        lib, st, g = L.get_lib(), _stream(), self.group
        ps = self._p2p_desc(x.shape[0], lr, since_fired, act_freq)
        n = self.group.world
        link = (n - 1) / n * 8 * self.d * self.F          # bytes pulled over NVLink per rank: both gradient matrices, (N-1)/N of the owned slice x N peers

        def rs():
            g.barrier(ps)
            L.check(lib.pb_p2p_reduce_scatter(C.byref(ps), st), "pb_p2p_reduce_scatter")

        def adam():
            g.barrier(ps)
            L.check(lib.pb_p2p_adam_allgather(C.byref(ps), st), "pb_p2p_adam_allgather")
            g.barrier(ps)
        return [("p2p barrier + reduce-scatter (peer loads over NVLink)", rs, dict(nvlink_bytes=link, ncu=r"k_p2p_reduce_scatter")),
                ("p2p barrier + sharded Adam + all-gather (peer stores) + barrier", adam,
                 dict(bytes=60 * self.d * self.F // n, nvlink_bytes=(n - 1) / n * (8 if self.W_encT_lo is None else 12) * self.d * self.F,
                      ncu=r"k_p2p_adam_allgather"))]     # pushed per rank: its W_dec and W_encT rows (+ the tf32 residual plane of the dense encoder) to N-1 peers
