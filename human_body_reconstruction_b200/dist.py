"""Data parallelism for the training step: one process per GPU, rays sharded across ranks, parameters
replicated, ONE flat gradient buffer per module all-reduced (averaged) over NCCL/NVLink inside
`loss.backward()` -- so an unchanged trainer (train_hash2.py:226-228: backward, then optimiser steps) sees
reduced gradients.  The reference has no counterpart (it wraps only the MLP in nn.DataParallel); this is
SURVEY section 8(e).

Two exchanges are provided: `GradAllReduce` (NCCL calls, below) and `PeerGradAllReduce` (ONE kernel of this
package over NVLink peer memory / NVLS multicast, csrc/comm.cu; the default of `attach_grad_allreduce`).

Mechanics (class _GradExchange): `HashEncoder` / `MLP_3D` accumulate into ONE persistent flat gradient buffer each -- (L,T,F) /
(14227,) -- that is zeroed once per backward pass however many autograd nodes feed it (a hierarchical render runs the field
twice); the last backward node of a module publishes its buffer (the encoder in level chunks, each as soon as its
scatter-add kernel has been enqueued) and the exchange of a published piece may start right there, overlapping what is
left of the backward; an end-of-backward engine callback reduces the rest, makes the compute stream wait, and only then
hands the buffers to `.grad`.  MSE is a mean over the LOCAL batch, so the average over ranks equals the single-process
gradient of the concatenated batch.  The modules' side of this protocol -- what every autograd node of HashEncoder /
MLP_3D does with or without an exchange attached -- is `node_params` and `ParamGrad`, below `_GradExchange`.
"""
from __future__ import annotations

import os
from typing import Iterable, List

import torch
import torch.distributed as dist
from torch.autograd import Variable


def init_from_env(backend: str | None = None) -> tuple[int, int]:
    """Initialises torch.distributed from RANK/WORLD_SIZE/MASTER_* (torchrun) and pins the CUDA device.
    Returns (rank, world)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world


class _GradExchange:
    """One backward pass = one SESSION.  The native modules (HashEncoder, MLP_3D) talk to the reducer installed in their
    `_dp` attribute through four calls:

        note_forward(m)            in the autograd forward, when gradients will be wanted (counts the backward nodes to expect;
                                   the first one of a step also starts zeroing the persistent buffers on a side stream)
        buf, last = enter_backward(m)   in every backward node: the module's persistent flat gradient buffer -- zeroed ONCE
                                   per session, so several passes through the same module (coarse + fine render,
                                   vol_renderer.py:220,242) ACCUMULATE into it -- and whether this is the last node expected
        publish(m, piece)          by the last node only, per finished piece (level chunk): may start that piece's exchange
        (the node returns None for the parameter gradients)

    and an autograd-engine end-of-backward callback reduces whatever was not published, makes the compute stream wait for
    the exchange and only then hands the buffers to the parameters' `.grad` (assigned, or added if the caller keeps
    gradients across backward calls).  Nothing is ever returned to AccumulateGrad while a collective may still write it, and
    every buffer is reduced exactly once per backward however many autograd nodes fed it."""

    def __init__(self, modules, group=None, average: bool = True):
        self.group, self.average = group, average
        self.modules = list(modules)
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self._fwd = {id(m): 0 for m in self.modules}
        self._pub = {id(m): [] for m in self.modules}        # published (offset, n) ranges of the module's buffer
        self._touched = set()                                 # modules that ran a backward node in this session
        self._active = False
        self._prezero = None                                  # event of a zero-fill running on the side stream
        self._zero_stream = None
        self.bytes_reduced = 0
        self.sessions = 0
        for m in self.modules:
            if getattr(m, "_dp", None) is not None:
                raise RuntimeError("module already has a gradient exchange attached")
            m._dp = self

    # -- to be provided -----------------------------------------------------------------------------------------
    def _buffer(self, m) -> torch.Tensor:                     # persistent flat gradient buffer of module m
        raise NotImplementedError

    def _reduce(self, m, offset: int, n: int):                # start the exchange of floats [offset, offset+n) of m's buffer
        raise NotImplementedError

    def _reduce_all(self) -> bool:                            # optional: one exchange for everything; True if done
        return False

    def _join(self):                                          # compute stream waits for every exchange started
        pass

    # above this many sample points per pass the table backward is not chunked: the step is long against the all-reduce
    # (2^17 rays x 128 samples: 11.7 ms against 0.2 ms) and every extra chunk re-reads the whole d(feature) tensor
    CHUNK_MAX_POINTS = 1 << 21

    def level_chunks(self, m, L: int, n_points: int = 0):
        """[(l0, l1), ...]: the level ranges the last table backward of a pass runs and publishes in.  `chunks` may be a
        count (equal level ranges) or a list of inner level boundaries, e.g. [4, 8, 12, 14] -> [0,4) [4,8) [8,12) [12,14)
        [14,16): all levels carry the same bytes, but the scatter-add of a coarse level costs a fraction of a fine one's,
        so early cheap chunks put bytes on the wire while most of the scatter-add is still to come."""
        c = self.chunks(m)
        if n_points > self.CHUNK_MAX_POINTS:
            return [(0, L)]
        if isinstance(c, (list, tuple)):
            b = [0] + sorted(int(v) for v in c if 0 < int(v) < L) + [L]
            return [(b[i], b[i + 1]) for i in range(len(b) - 1) if b[i + 1] > b[i]]
        n = max(1, min(L, int(c)))
        step = -(-L // n)
        return [(l0, min(L, l0 + step)) for l0 in range(0, L, step)]

    def chunks(self, m) -> int:                               # pieces the last backward node of m should publish in
        return 1

    def stream_plan(self, m, L: int, n_points: int = 0):
        """Level chunks for a STREAMED exchange of the last table backward (one producer launch + one exchange launch running
        side by side, PeerGradAllReduce(streamed=True)), or None: the caller then runs level_chunks() launch by launch."""
        return None

    # -- module side ----------------------------------------------------------------------------------------------
    def remove(self):
        for m in self.modules:
            if getattr(m, "_dp", None) is self:
                m._dp = None

    def _zero_buffers(self):
        for m in self.modules:
            self._buffer(m).zero_()

    def _detach_aliases(self):
        """A parameter whose .grad still IS the persistent buffer (the caller kept gradients: zero_grad(set_to_none=False)
        or gradient accumulation) gets its own copy before the buffer is reused."""
        for m in self.modules:
            for p, v in m._dp_param_views(self._buffer(m)):
                if p.grad is not None and p.grad.data_ptr() == v.data_ptr():
                    p.grad = p.grad.clone()

    def note_forward(self, m):
        first = not self._active and self._prezero is None and not any(self._fwd.values())
        self._fwd[id(m)] += 1
        if first and self._buffer(m).is_cuda:
            self._detach_aliases()
            cur = torch.cuda.current_stream()
            if self._zero_stream is None:
                self._zero_stream = torch.cuda.Stream()
            self._zero_stream.wait_stream(cur)                # everything that still reads last step's gradients is enqueued
            with torch.cuda.stream(self._zero_stream):
                self._zero_buffers()
                self._prezero = self._zero_stream.record_event()

    def _begin(self):
        if self._active:
            return
        self._active = True
        self.sessions += 1
        Variable._execution_engine.queue_callback(self._finish)
        if self._prezero is not None:
            torch.cuda.current_stream().wait_event(self._prezero)
            self._prezero = None
        else:
            self._detach_aliases()
            self._zero_buffers()

    def enter_backward(self, m):
        self._begin()
        k = id(m)
        self._touched.add(k)
        self._fwd[k] = max(self._fwd[k] - 1, 0)
        return self._buffer(m), self._fwd[k] == 0

    def publish(self, m, piece: torch.Tensor):
        buf = self._buffer(m)
        off = (piece.data_ptr() - buf.data_ptr()) // buf.element_size()
        n = piece.numel()
        if self._start_on_publish():
            self._reduce(m, off, n)
            self._pub[id(m)].append((off, n))

    def _start_on_publish(self) -> bool:
        return True

    def _gaps(self, m):
        total = self._buffer(m).numel()
        pos, out = 0, []
        for off, n in sorted(self._pub[id(m)]):
            if off > pos:
                out.append((pos, off - pos))
            pos = max(pos, off + n)
        if pos < total:
            out.append((pos, total - pos))
        return out

    def _finish(self):
        try:
            if self.world > 1:
                nothing = not any(self._pub.values())
                if not (nothing and self._reduce_all()):
                    for m in self.modules:
                        if id(m) not in self._touched:           # took no part in this backward (same on every rank)
                            continue
                        for off, n in self._gaps(m):
                            self._reduce(m, off, n)
                self._join()
            for m in self.modules:
                if id(m) not in self._touched:
                    continue
                for p, v in m._dp_param_views(self._buffer(m)):
                    if not p.requires_grad:
                        continue
                    if p.grad is None:
                        p.grad = v
                    else:
                        p.grad.add_(v)
        finally:
            self._active = False
            self._touched = set()
            for k in self._fwd:
                self._fwd[k] = 0
                self._pub[k] = []


def node_params(*modules) -> list:
    """The parameters an autograd node of these modules is applied with.  Under no_grad they are passed detached: the node
    decides from needs_input_grad, which follows requires_grad and not the grad mode, whether to count itself with the
    exchange or pre-zero a table gradient buffer, and no backward would ever read either."""
    ps = [p for m in modules for p in m._dp_params()]
    return ps if torch.is_grad_enabled() else [p.detach() for p in ps]


class ParamGrad:
    """One autograd node's gradient of one module's parameters (HashEncoder tables or MLP_3D), created in the node's
    forward and kept on ctx.  `wanted`: whether the node's parameter inputs need a gradient.  When they do, the forward
    notes the node with the module's exchange or, without one, starts the module's side-stream pre-zero
    (HashEncoder._zeroed_grad_async).  In the backward:

        buffer()            the flat buffer to accumulate into: the exchange's, the pre-zeroed one or fresh zeros
        stream_plan(n)      the level chunks of a streamed exchange (only the last table node under one), else None
        scatter_table(...)  the table's scatter-add schedule: one level range, level chunks or a streamed exchange
        complete(piece)     a finished piece (default: the whole buffer); the last node under an exchange publishes it
        grads()             what the node returns to autograd for the parameters; ends the node's backward"""

    def __init__(self, m, wanted: bool):
        self.m, self.wanted = m, bool(wanted)
        self.exchange = m._dp if wanted else None
        self.buf, self.last, self._pre = None, False, None
        self._flat = m._flat                  # the storage the forward ran with (its _flat_table() / _flat_params())
        if self.exchange is not None:
            self.exchange.note_forward(m)
        elif wanted and hasattr(type(m), "_zeroed_grad_async"):
            self._pre = m._zeroed_grad_async()

    def buffer(self) -> torch.Tensor:
        if self.buf is None:
            if self.exchange is not None:
                self.buf, self.last = self.exchange.enter_backward(self.m)
            elif self._pre is not None:
                self.buf, ev = self._pre
                self._pre = None
                torch.cuda.current_stream().wait_event(ev)
            else:
                self.buf = torch.zeros_like(self._flat)
        return self.buf

    def stream_plan(self, n_points: int):
        if self.exchange is None:
            return None
        self.buffer()
        return self.exchange.stream_plan(self.m, self.m.L, n_points) if self.last else None

    def complete(self, piece: torch.Tensor | None = None):
        if self.exchange is not None and self.last:
            self.exchange.publish(self.m, self.buf if piece is None else piece)

    def grads(self) -> tuple:
        buf, self.buf, self.last = self.buf, None, False          # a retained graph's next backward starts afresh
        if self.exchange is not None or not self.wanted:
            return (None,) * len(self.m._dp_params())             # the exchange hands its buffer to .grad
        return tuple(self.m._grad_views(buf))

    def scatter_table(self, run, n_points: int, stream=None, after_first=None, mlp: "ParamGrad | None" = None,
                      mlp_stream=None):
        """Enqueues the table gradient.  run(g, l0, l1): the scatter-add of levels [l0, l1) into g.  One level range,
        except in the last node under an exchange: level chunks, each published as soon as its scatter-add is enqueued,
        so its all-reduce overlaps the next chunk's scatter-add.  With `stream` and a streamed exchange (stream_plan):
        stream(g, chunks, done) enqueues ONE scatter-add launch that finishes the chunks in order and returns the count a
        chunk's done word reaches, and the exchange is ONE launch beside it on the exchange's side stream.  That launch
        also carries the gradient of `mlp` when it is the same exchange's last MLP node, once `mlp_stream` (the stream
        finishing it, or None) gets there.  after_first() runs behind the first chunk's scatter-add, or behind the
        streamed exchange's launch."""
        g = self.buffer()
        plan = self.stream_plan(n_points) if stream is not None else None
        if plan is not None:
            ev_pre = torch.cuda.current_stream().record_event()
            need = stream(g, plan, self.exchange.done)
            with_mlp = mlp is not None and mlp.exchange is self.exchange and mlp.last
            ev_mlp = mlp_stream.record_event() if (mlp_stream is not None and with_mlp) else None
            self.exchange.exchange_streamed(plan, need, after=(ev_pre, ev_mlp), include_mlp=with_mlp)
            if with_mlp:
                mlp.last = False                                  # published by that launch
            if after_first is not None:
                after_first()
            return
        L = self.m.L
        for l0, l1 in (self.exchange.level_chunks(self.m, L, n_points) if self.last else [(0, L)]):
            run(g, l0, l1)
            if l0 == 0 and after_first is not None:
                after_first()
            self.complete(g[l0:l1])


class GradAllReduce(_GradExchange):
    """`GradAllReduce(encoder, mlp)`: the exchange as asynchronous torch.distributed all-reduces (NCCL; gloo on CPU ranks)
    on persistent flat gradient buffers.  Detach with `.remove()`."""

    def __init__(self, *modules, group=None, average: bool = True, chunks: int = 1):
        super().__init__(modules, group=group, average=average)
        self._bufs = {}
        self._pending: List = []
        self._chunks = int(chunks)

    def chunks(self, m) -> int:
        return max(1, int(getattr(m, "_grad_chunks", 0) or self._chunks))

    def _buffer(self, m):
        b = self._bufs.get(id(m))
        t = m._dp_template()
        if b is None or b.device != t.device or b.shape != t.shape:
            b = self._bufs[id(m)] = torch.zeros_like(t)
        return b

    def _reduce(self, m, offset, n):
        if not dist.is_initialized() or self.world == 1:
            return
        flat = self._buffer(m).view(-1)[offset:offset + n]
        op = dist.ReduceOp.SUM
        if self.average:
            if dist.get_backend(self.group) == "nccl":
                op = dist.ReduceOp.AVG                        # averaging inside the collective: no extra pass over the buffer
            else:
                flat.div_(self.world)
        self._pending.append(dist.all_reduce(flat, op=op, group=self.group, async_op=True))
        self.bytes_reduced += n * flat.element_size()

    def _join(self):
        for w in self._pending:
            w.wait()                       # compute stream waits on the collective's stream; no host sync for CUDA tensors
        self._pending.clear()


class PeerGradAllReduce(_GradExchange):
    """`PeerGradAllReduce(encoder, mlp)`: the same contract, but the exchange is ONE kernel over NVLink peer memory
    (csrc/comm.cu) instead of NCCL calls.  The two modules' gradient buffers are slices of one persistent peer-mapped region
    [table (L,T,F) | MLP parameters]; the scatter-add of the hash-grid backward and the MLP gradient reduction write
    straight into it, and hbr_allreduce_peer runs on the compute stream behind them (capturable in the step's CUDA
    graph).  Every rank ends with bit-identical averaged gradients.  A failed exchange (flag-barrier timeout) raises at
    the next step's end of backward instead of letting the optimiser run on."""

    def __init__(self, encoder, mlp, group=None, average: bool = True, transport: str = "ipc", ctas: int = 0,
                 overlap: bool = False, chunks: int = 2, streamed: bool = False):
        """overlap=False: one all-reduce of the whole region behind the backward pass.  overlap=True: the LAST table backward
        of the pass runs in `chunks` level chunks and every published piece (the MLP gradient first, then each level chunk)
        is all-reduced at once by a small grid (`ctas`, default 32) on a high-priority side stream while the next chunk's
        scatter-add still runs on the compute stream.  streamed=True (with overlap): the chunks are not separate launches --
        ONE scatter-add launch finishes them in order and counts finished CTAs per chunk (hbr_hash_encode_bwd*_stream), ONE
        exchange launch beside it (hbr_allreduce_peer_stream) sends each chunk as soon as its count is complete on every
        rank: no launch gaps, no per-chunk tails, and the flag barriers of a chunk hide behind the next chunk's scatter-add."""
        from .peer import PeerRegion
        n_tab = encoder.L * encoder.T * encoder.F
        n_mlp = mlp._flat_params().numel()
        off = -(-n_tab // 4) * 4
        self.region = PeerRegion(off + n_mlp, group=group, transport=transport)
        self.overlap = overlap
        self.ctas = ctas if ctas > 0 else (32 if overlap else 0)
        self._nchunks = [int(v) for v in chunks] if isinstance(chunks, (list, tuple)) else int(chunks)
        self._enc, self._mlp = encoder, mlp
        encoder._flat_table()
        self._slices = {id(encoder): self.region.tensor[:n_tab].view(encoder.L, encoder.T, encoder.F),
                        id(mlp): self.region.tensor[off:off + n_mlp]}
        self._side = torch.cuda.Stream(device=self.region.device, priority=-1) if overlap else None
        self._base = self.region.tensor.data_ptr()
        self._side_used = False
        self.streamed = bool(streamed and overlap)
        self._done = torch.zeros(64, dtype=torch.int32, device=self.region.device)   # finished CTAs per level chunk
        super().__init__([encoder, mlp], group=group, average=average)

    def remove(self):
        super().remove()

    def chunks(self, m) -> int:
        return self._nchunks if (self.overlap and m is self._enc) else 1

    def _scale(self):
        return 1.0 / self.world if self.average else 1.0

    def _buffer(self, m):
        return self._slices[id(m)]

    def _zero_buffers(self):
        self.region.tensor.zero_()                            # one memset over [table | MLP]
        if self.streamed:
            self._done.zero_()

    def _start_on_publish(self) -> bool:
        return self.overlap

    def stream_plan(self, m, L: int, n_points: int = 0):
        if not self.streamed or m is not self._enc or n_points > self.CHUNK_MAX_POINTS or n_points <= 0:
            return None
        ch = self.level_chunks(m, L, n_points)
        return ch if len(ch) > 1 else None

    @property
    def done(self) -> torch.Tensor:
        return self._done

    def exchange_streamed(self, chunks, need: int, after=(), include_mlp: bool = False):
        """Called by the last table backward right AFTER it has enqueued the producer (ops.hash_encode_bwd*_lm or *_stream with
        `chunks` and self.done) on the compute stream; `need` = the count a chunk's done word reaches when the chunk is
        complete (ops.hash_bwd_lm_ctas / hash_bwd_stream_tiles).  Enqueues the exchange of [MLP gradient (include_mlp: it is
        complete once the events in `after` have fired) | level chunks] on the side stream, which waits for `after` only --
        not for the scatter-add it runs beside."""
        enc, mlp = self._enc, self._mlp
        per_level = enc.T * enc.F
        tiles = int(need)
        pieces = []
        if include_mlp:
            off = (self._slices[id(mlp)].data_ptr() - self._base) // 4
            pieces.append((off, self.region.n - off, 0, 0))
            self._pub[id(mlp)].append((0, self._slices[id(mlp)].numel()))
        for c, (l0, l1) in enumerate(chunks):
            pieces.append((l0 * per_level, (l1 - l0) * per_level, tiles, c))
        self._pub[id(enc)].append((0, enc.L * per_level))
        for ev in after:
            if ev is not None:
                self._side.wait_event(ev)
        with torch.cuda.stream(self._side):
            self.region.all_reduce_stream(pieces, self._done, scale=self._scale(), ctas=self.ctas)
        self._side_used = True
        self.bytes_reduced += 4 * sum(p[1] for p in pieces)

    def _reduce(self, m, offset, n):
        off = (self._buffer(m).data_ptr() - self._base) // 4 + offset
        lo = off // 4 * 4                                     # whole float4s; the slack belongs to padding or a piece reduced
        n4 = -(-(off + n - lo) // 4) * 4                      # in the same call sequence on every rank
        if self._side is not None:
            cur = torch.cuda.current_stream()
            self._side.wait_stream(cur)                       # the piece's producer kernel has been enqueued on `cur`
            with torch.cuda.stream(self._side):
                self.region.all_reduce(n=n4, scale=self._scale(), ctas=self.ctas, offset=lo)
            self._side_used = True
        else:
            self.region.all_reduce(n=n4, scale=self._scale(), ctas=self.ctas, offset=lo)
        self.bytes_reduced += n4 * 4

    def _reduce_all(self) -> bool:
        if self._side is not None:
            return False
        self.region.all_reduce(scale=self._scale(), ctas=self.ctas)
        self.bytes_reduced += self.region.n * 4
        return True

    def _join(self):
        if self._side_used:
            torch.cuda.current_stream().wait_stream(self._side)
            self._side_used = False
        self.region.raise_if_failed()                         # the status word copied out at the end of the PREVIOUS step
        self.region.poll_status()


def attach_grad_allreduce(encoder, mlp, group=None, kind: str = "auto", **peer_kw):
    """The gradient exchange for `world` > 1: kind "peer" = PeerGradAllReduce, "nccl" = GradAllReduce, "auto" = peer
    when every rank can set it up (CUDA ranks of one node), else NCCL.  Peer transport "auto": 2 ranks exchange through
    plain peer loads/stores over CUDA-IPC mappings (measured 0.130 ms for 67 MB against 0.153 ms NCCL and 0.21 ms
    multicast); more ranks reduce inside the NVSwitch through an NVLS multicast mapping when torch's symmetric memory
    offers one (8 ranks: 0.184 ms against 0.240 ms peer loads/stores and 0.245 ms NCCL)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return None
    if kind == "nccl" or not torch.cuda.is_available() or dist.get_backend(group) != "nccl":
        return GradAllReduce(encoder, mlp, group=group, chunks=int(peer_kw.get("chunks", 1)) if kind == "nccl" else 1)
    world = dist.get_world_size(group)
    kw = dict(peer_kw)
    kw.setdefault("overlap", True)        # launch-per-chunk form, measured best at 4 096 rays/GPU: 2 level chunks, 32 CTAs on
    kw.setdefault("chunks", 2)            # the side stream (W=8: 0.656 ms/step against 0.712 behind the backward, 0.671 with 4)
    if kw.get("streamed", None) is None:
        # W >= 3 (NVLS multicast): one scatter-add launch + one exchange launch side by side, 4 equal level chunks
        # (W=8, 4 096 rays/GPU: 0.591 ms/step; 3 chunks 0.596; [6,10,13] 0.598; [6,9,12,14] 0.606; a launch pair per chunk 0.639).
        # W = 2 (peer loads/stores, which take SMs and L2 bandwidth from the scatter-add they run beside): a launch pair
        # per chunk, 2 chunks: 0.639 ms/step against 0.688 streamed
        kw["streamed"] = world > 2
        if "chunks" not in peer_kw:
            kw["chunks"] = 4 if world > 2 else 2
    if kw.get("transport", "auto") == "auto":
        kw["transport"] = "ipc" if world == 2 else "symm"
    red, err = None, None
    try:
        red = PeerGradAllReduce(encoder, mlp, group=group, **kw)
    except Exception as e:                                   # e.g. no peer access between the devices
        err = e
    ok = torch.tensor([1 if red is not None else 0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
    if int(ok.item()) == 1:
        return red
    if red is not None:
        red.remove()
    if kind == "peer":
        raise RuntimeError(f"peer-memory all-reduce unavailable on at least one rank: {err!r}")
    return GradAllReduce(encoder, mlp, group=group)


def broadcast_parameters(encoder, mlp, src: int = 0, group=None):
    """Every rank takes rank `src`'s hash tables and MLP parameters (the unchanged trainer does not seed: each process
    initialised its own).  Two broadcasts of the flat buffers."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    with torch.no_grad():
        dist.broadcast(encoder._flat_table(), src=src, group=group)
        dist.broadcast(mlp._flat_params(), src=src, group=group)


def attach_small_params(params, group=None, src: int = 0):
    """Parameters that live outside the two flat gradient buffers -- SDF mode's VarModel.b (helper.py:13-21), one float --:
    every rank takes rank `src`'s value now, and a post-accumulate hook averages the gradient over the ranks inside
    loss.backward() (one tiny all-reduce per parameter; the table and MLP gradients keep their own exchange).  Idempotent."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return []
    done = []
    for p in params:
        if getattr(p, "_hbr_dp_hook", None) is not None:
            continue
        with torch.no_grad():
            dist.broadcast(p.data, src=src, group=group)

        def hook(q, group=group):
            if q.grad is not None:
                dist.all_reduce(q.grad, op=dist.ReduceOp.SUM, group=group)
                q.grad.div_(dist.get_world_size(group))

        p._hbr_dp_hook = p.register_post_accumulate_grad_hook(hook)
        done.append(p)
    return done


def auto_attach(encoder, mlp, group=None, extra=()):
    """launch_rank.py's zero-edit route (HBR_AUTO_DP=1): called by Volume_Renderer at its first native vol_render of a
    process that belongs to a process group -- broadcast rank 0's parameters, attach the gradient exchange (once).
    extra: further small parameters of the step (SDF mode's VarModel), see attach_small_params."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return None
    attach_small_params(extra, group)
    if getattr(encoder, "_dp", None) is not None:
        return encoder._dp
    broadcast_parameters(encoder, mlp, 0, group)
    return attach_grad_allreduce(encoder, mlp, group=group)


def shard_rays(n_rays: int, rank: int, world: int) -> slice:
    """Rank r takes rays [r*n/world, (r+1)*n/world) (SURVEY 8e)."""
    per = n_rays // world
    return slice(rank * per, (rank + 1) * per if rank < world - 1 else n_rays)


def slab_range(res: int, rank: int, world: int) -> tuple[int, int]:
    """Planes [i0, i1) of axis 0 of the density grid owned by `rank` (nerf2mesh grid sharding)."""
    base, rem = divmod(res, world)
    i0 = rank * base + min(rank, rem)
    return i0, i0 + base + (1 if rank < rem else 0)


def allgather_counts(counts: Iterable[int]) -> list[list[int]]:
    """Per-rank (vertices, triangles) -> list over ranks; exclusive prefix gives each rank's output offsets."""
    t = torch.tensor(list(counts), dtype=torch.int64)
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return [t.tolist()]
    if dist.get_backend() == "nccl":
        t = t.cuda()
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [o.tolist() for o in out]
