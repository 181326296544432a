"""Multi-GPU execution: slab decomposition of the outermost dimension with per-pass halo exchange.

The reference scales across devices by cutting the *operator pipeline* in two and streaming whole
fields through SMI channels (``split_sdfg``, ``stencilflow/sdfg_generator.py:680-1000``;
``bin/run_distributed_program.py``); its remote streams run concurrently with the compute pipeline
(``sdfg_generator.py:846-853``).  On a box of NVLink-connected GPUs the natural decomposition is
spatial instead: rank g owns planes ``[g*N/G, (g+1)*N/G)`` of the outermost dimension (i for 3-D, j for
2-D programs); row-major layout makes every halo one contiguous block.  A field that a later pass
reads across the slab boundary reaches the neighbours' halo planes in one of two ways:

* **in-kernel push** (streamed passes): the producing kernel stores the few planes next to a slab
  boundary a second time, straight into the neighbour's buffer (peer stores over NVLink on IPC-mapped
  memory) -- the transfer rides along with the pass tile by tile, nothing is copied afterwards;
* **copy push** (one-operator kernels): peer ``cudaMemcpyAsync`` of the edge planes on a separate
  communication stream, ordered behind the producing launch by an event.

Either way the data path is flag-ordered, with no host synchronisation and no collective (``ExchangePlan``):
after the push a counter is raised in the neighbour's memory (``cuStreamWriteValue32``) and the
neighbour's consumer launch waits for it (``cuStreamWaitValue32``, >=); a second counter per
neighbour publishes how far that neighbour's own launches have come, which is what a pusher waits
for before it overwrites halo planes a launch over there may still be reading.  Exchange
participation is a property of the *plan*, identical on every rank (a rank with a one-sided reach
still receives, still counts), and results are bit-identical to the single-GPU run because every
cell is computed by the same instruction sequence.

One process per GPU.  Rendezvous (exchange of IPC handles, barriers, max-reduction of timings) goes
through a tiny ``Comm`` interface: ``SocketComm`` (plain TCP on 127.0.0.1, no dependencies) or
``TorchComm`` (``torch.distributed``/gloo, which is how ``torchrun`` launches ``bench.py``).  Neither
touches device memory or the data path.
"""

import os
import pickle
from typing import Dict, List, Optional

import numpy as np


class Slab:
    """Ownership of the slab axis for one rank: owned planes [begin, end), allocated planes
    [alloc_begin, alloc_end) = owned + halo, clipped to the domain."""

    def __init__(self, rank, world, n, halo):
        if n < world:
            raise ValueError("cannot split {} planes over {} ranks".format(n, world))
        self.rank, self.world, self.n, self.halo = rank, world, n, halo
        self.begin = (n * rank) // world
        self.end = (n * (rank + 1)) // world
        self.alloc_begin = max(0, self.begin - halo)
        self.alloc_end = min(n, self.end + halo)
        if world > 1 and (self.end - self.begin) < halo:
            raise ValueError("slab of {} planes is thinner than the halo {}".format(self.end - self.begin, halo))

    @staticmethod
    def of_rank(rank, world, n, halo):
        return Slab(rank, world, n, halo)

    def __repr__(self):
        return "Slab(rank {}/{}: own [{}, {}), alloc [{}, {}))".format(
            self.rank, self.world, self.begin, self.end, self.alloc_begin, self.alloc_end)


class HaloSend:
    """After launch ``launch``: planes [src_begin, src_end) of ``field`` go to rank ``peer``."""

    def __init__(self, launch, field, peer, src_begin, src_end):
        self.launch, self.field, self.peer = launch, field, peer
        self.src_begin, self.src_end = src_begin, src_end

    def __repr__(self):
        return "HaloSend(after launch {}: {}[{}:{}] -> rank {})".format(
            self.launch, self.field, self.src_begin, self.src_end, self.peer)


def launch_reach(lowered, launch_index):
    """(back, fwd): how many planes below / above its output range a launch reads along the slab
    axis, per field it reads: {field: (back, fwd)}."""
    l = lowered.launches[launch_index]
    program = lowered.program
    axis = lowered.slab_axis
    reach = {}
    if axis is None:
        return reach
    it = "ijk"[axis]
    if l.family == "streamed":
        for f, (b, fw) in l.info["reach"].items():
            reach[f] = (b, fw)
        return reach
    op = next(o for o in program.ops if o.name == l.ops[0])
    pos = "ijk".index(it)
    for f in l.reads:
        if it not in program.fields[f].dims:
            continue
        lo = hi = 0
        for off in op.offsets3(f):
            if off[pos] is not None:
                lo, hi = min(lo, off[pos]), max(hi, off[pos])
        reach[f] = (-lo, hi)
    return reach


def halo_depth(lowered):
    """Planes of halo every slab-decomposed buffer is allocated with."""
    h = 0
    for idx in range(len(lowered.launches)):
        for (b, f) in launch_reach(lowered, idx).values():
            h = max(h, b, f)
    return h


def total_reach(lowered):
    """Planes below / above the owned range that the *whole program* reaches for along the slab
    axis: the halo a rank needs to run all its launches without any exchange, recomputing the
    intermediate halo planes itself (what the overlapped host-array call does)."""
    need_back = need_fwd = 0
    acc = {}                       # field -> (back, fwd) still needed of it beyond the owned range
    for idx in range(len(lowered.launches) - 1, -1, -1):
        l = lowered.launches[idx]
        b0 = max([acc.get(w, (0, 0))[0] for w in l.writes] + [0])
        f0 = max([acc.get(w, (0, 0))[1] for w in l.writes] + [0])
        for f, (b, fw) in launch_reach(lowered, idx).items():
            old = acc.get(f, (0, 0))
            acc[f] = (max(old[0], b0 + b), max(old[1], f0 + fw))
            need_back, need_fwd = max(need_back, acc[f][0]), max(need_fwd, acc[f][1])
    return max(need_back, need_fwd)


def halo_schedule(lowered, slab: Slab) -> List["HaloSend"]:
    """Which planes this rank must push to which neighbour after which launch (``ExchangePlan.for_rank``).

    Field F written by launch l and read by a later launch with reach (back, fwd) along the slab
    axis: the upper neighbour needs my top ``back`` planes as its lower halo, the lower neighbour my
    bottom ``fwd`` planes as its upper halo.  Program inputs are loaded with their halos and never
    exchanged."""
    return ExchangePlan(lowered).for_rank(slab)


class ExchangePlan:
    """What the launches of a plan exchange across slab boundaries, and the counter values that order
    it.  Everything here is derived from the plan alone, so every rank computes the same object; only
    ``for_rank`` looks at who has which neighbour.

    ``up[idx]`` / ``down[idx]``: ``[(field, planes)]`` -- after launch ``idx`` the top ``planes`` owned
    planes of ``field`` go up (to rank + 1, as its lower halo), resp. the bottom ``planes`` go down.
    Channel counters: the k-th launch with an ``up`` entry raises the receiver's *from-below* counter
    to ``rep * len(up_events) + k + 1`` in repetition ``rep`` of the program; likewise *from-above*.
    Progress counter: after launch ``idx`` of repetition ``rep`` a rank tells both neighbours
    ``rep * n_launches + idx + 1`` (only after launches somebody waits for, ``progress_points``)."""

    def __init__(self, lowered, storage=None):
        self.n = len(lowered.launches)
        self.up = [[] for _ in range(self.n)]
        self.down = [[] for _ in range(self.n)]
        storage = storage or {}
        if lowered.slab_axis is not None:
            reach = [launch_reach(lowered, idx) for idx in range(self.n)]
            for idx, l in enumerate(lowered.launches):
                for field in l.writes:
                    back = fwd = 0
                    for later in range(idx + 1, self.n):
                        r = reach[later].get(field)
                        if r:
                            back, fwd = max(back, r[0]), max(fwd, r[1])
                    if back:
                        self.up[idx].append((field, back))
                    if fwd:
                        self.down[idx].append((field, fwd))
        self.up_events = [idx for idx in range(self.n) if self.up[idx]]
        self.down_events = [idx for idx in range(self.n) if self.down[idx]]
        # before launch j: how many up / down events of this repetition must have arrived
        self.need_up = [sum(1 for e in self.up_events if e < j) for j in range(self.n)]
        self.need_down = [sum(1 for e in self.down_events if e < j) for j in range(self.n)]
        # write-after-read at the receiver: the halo planes of ``field`` (storage S) may only be
        # overwritten once every launch over there that read the previous content of S is done --
        # the last reader before ``idx`` in program order, wrapping into the previous repetition
        readers = {}
        for j, l in enumerate(lowered.launches):
            for f in l.reads:
                readers.setdefault(storage.get(f, f), set()).add(j)
        self.war = []                  # per launch: (repetition offset 0 / -1, launch index) or None
        for idx in range(self.n):
            last = None
            for (field, _) in self.up[idx] + self.down[idx]:
                rs = readers.get(storage.get(field, field), set())
                before = [j for j in rs if j < idx]
                after = [j for j in rs if j > idx]
                cand = (0, max(before)) if before else ((-1, max(after)) if after else None)
                if cand is not None and (last is None or cand > last):
                    last = cand
            self.war.append(last)
        self.progress_points = sorted({w[1] for w in self.war if w is not None})

    def arrival_value(self, channel, rep, idx):
        events = self.up_events if channel == "up" else self.down_events
        return rep * len(events) + events.index(idx) + 1

    def wait_values(self, rep, idx):
        """(from-below, from-above) counter values launch ``idx`` of repetition ``rep`` needs (0 = none)."""
        lo = rep * len(self.up_events) + self.need_up[idx] if self.need_up[idx] else 0
        hi = rep * len(self.down_events) + self.need_down[idx] if self.need_down[idx] else 0
        return lo, hi

    def war_value(self, rep, idx):
        """Progress a neighbour must have reported before launch ``idx`` of repetition ``rep`` pushes
        into its halo planes (0 = nothing to wait for)."""
        w = self.war[idx]
        if w is None:
            return 0
        return max(0, (rep + w[0]) * self.n + w[1] + 1)

    def for_rank(self, slab: Slab):
        """``[(launch, field, peer, src_begin, src_end)]`` this rank pushes, as :class:`HaloSend`."""
        sends = []
        if slab.world == 1:
            return sends
        for idx in range(self.n):
            for (field, back) in self.up[idx]:
                if slab.rank + 1 < slab.world:
                    sends.append(HaloSend(idx, field, slab.rank + 1, slab.end - back, slab.end))
            for (field, fwd) in self.down[idx]:
                if slab.rank > 0:
                    sends.append(HaloSend(idx, field, slab.rank - 1, slab.begin, slab.begin + fwd))
        return sends


# ------------------------------------------------------------------------------------ rendezvous


class Comm:
    rank = 0
    world = 1

    def allgather(self, obj):
        return [obj]

    def barrier(self):
        pass

    def max_float(self, x):
        return x

    def close(self):
        pass


class TorchComm(Comm):
    """``torch.distributed`` (gloo) as rendezvous: reads RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT."""

    def __init__(self, backend="gloo"):
        import torch.distributed as dist
        self.dist = dist
        self.owns = not dist.is_initialized()
        if self.owns:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group(backend=backend)
        self.rank = dist.get_rank()
        self.world = dist.get_world_size()

    def allgather(self, obj):
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def barrier(self):
        self.dist.barrier()

    def max_float(self, x):
        return max(self.allgather(float(x)))

    def close(self):
        if self.owns and self.dist.is_initialized():
            self.dist.destroy_process_group()


class SocketComm(Comm):
    """Rendezvous over plain TCP on one box, no dependencies: rank 0 listens on
    ``MASTER_ADDR:SFB200_COMM_PORT`` (default ``MASTER_PORT + 1``), the other ranks connect; every
    collective is an all-gather of pickled objects through rank 0.  Carries a few hundred bytes (IPC
    handles, timings) -- the data path is NVLink."""

    def __init__(self, rank=None, world=None, addr=None, port=None, timeout=120.0):
        import socket
        import time
        self.rank = int(os.environ["RANK"]) if rank is None else rank
        self.world = int(os.environ["WORLD_SIZE"]) if world is None else world
        addr = addr or os.environ.get("MASTER_ADDR", "127.0.0.1")
        port = int(port or os.environ.get("SFB200_COMM_PORT", 0) or int(os.environ.get("MASTER_PORT", "29500")) + 1)
        self.peers = []
        self.sock = None
        if self.world == 1:
            return
        if self.rank == 0:
            srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
            srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
            srv.bind((addr, port))
            srv.listen(self.world)
            srv.settimeout(timeout)
            conns = {}
            while len(conns) < self.world - 1:
                c, _ = srv.accept()
                c.settimeout(timeout)
                c.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
                r = pickle.loads(self._recv(c))
                conns[r] = c
            srv.close()
            self.peers = [conns[r] for r in range(1, self.world)]
        else:
            deadline = time.time() + timeout
            while True:
                try:
                    self.sock = socket.create_connection((addr, port), timeout=timeout)
                    break
                except OSError:
                    if time.time() > deadline:
                        raise
                    time.sleep(0.05)
            self.sock.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
            self._send(self.sock, pickle.dumps(self.rank))

    @staticmethod
    def _send(sock, payload):
        sock.sendall(len(payload).to_bytes(8, "little") + payload)

    @staticmethod
    def _recv(sock):
        def exactly(n):
            buf = bytearray()
            while len(buf) < n:
                chunk = sock.recv(n - len(buf))
                if not chunk:
                    raise ConnectionError("peer closed the rendezvous connection")
                buf += chunk
            return bytes(buf)
        return exactly(int.from_bytes(exactly(8), "little"))

    def allgather(self, obj):
        if self.world == 1:
            return [obj]
        if self.rank == 0:
            out = [obj] + [pickle.loads(self._recv(c)) for c in self.peers]
            payload = pickle.dumps(out)
            for c in self.peers:
                self._send(c, payload)
            return out
        self._send(self.sock, pickle.dumps(obj))
        return pickle.loads(self._recv(self.sock))

    def barrier(self):
        self.allgather(None)

    def max_float(self, x):
        return max(self.allgather(float(x)))

    def close(self):
        for c in self.peers + ([self.sock] if self.sock else []):
            try:
                c.close()
            except OSError:
                pass
        self.peers, self.sock = [], None


def make_comm():
    """The rendezvous of this launch: ``SFB200_COMM`` = ``socket`` (plain TCP, what ``bin/run_distributed_program.py``
    uses for the ranks it starts itself) or ``torch`` (``torch.distributed``/gloo -- the default under
    ``torchrun``, whose own store already owns ``MASTER_PORT``)."""
    kind = os.environ.get("SFB200_COMM", "torch" if "TORCHELASTIC_RUN_ID" in os.environ else "socket")
    return SocketComm() if kind == "socket" else TorchComm()


# ------------------------------------------------------------------------------------ device side


def _cuda_program_base():
    from .cuda_program import CudaProgram
    return CudaProgram


PEER_PUSH_DEFAULT = "0"


class SlabProgram:
    """A stencil program executed on this rank's slab.  Same execution interface as ``CudaProgram``
    (``execute``, ``launch_count``, ``plan``, ``buffers`` ...) plus slab-aware upload/download."""

    def __init__(self, stencil_file, comm: Comm, device=None, plan_options=None):
        from .cuda_program import CudaProgram
        from .kernel_chain_graph import KernelChainGraph
        from .stencil_op import make_program
        from . import planner
        self.comm = comm
        chain = KernelChainGraph(stencil_file)
        if plan_options is None:
            plan_options = planner.PlanOptions()
        # how the edge planes of a streamed pass reach the neighbours' halos: peer copies on the communication
        # streams behind the launch (default, the path one-operator kernels take too), or SFB200_PEER_PUSH=1:
        # the kernel stores them itself after each segment.  The in-kernel push overlaps the transfer with the
        # rest of the pass, but its kernel variant runs 6-15 % slower than the plain one (same loop, a less
        # lucky register assignment: 4.21-4.57 vs 3.96 ms per step at N = 4, profiles/r02d_push_kinds.txt)
        plan_options.peer_push = comm.world > 1 and os.environ.get("SFB200_PEER_PUSH", PEER_PUSH_DEFAULT) != "0"
        plan_options.cluster = 0            # a thread-block cluster is one GPU's
        probe = planner.plan_program(make_program(chain), options=plan_options)
        axis = probe.lowered.slab_axis
        if axis is None:
            raise ValueError("1-D programs do not shard")
        n = probe.program.shape3[axis]
        self.halo = halo_depth(probe.lowered)
        # buffers wide enough for the exchange-free host-array call (``__call__``) when that costs
        # little: the accumulated reach of the program, at most a quarter of the thinnest slab
        wide = total_reach(probe.lowered)
        if os.environ.get("SFB200_SLAB_WIDE_HALO", "1") != "0" and wide <= (n // comm.world) // 4:
            self.halo = max(self.halo, wide)
        self.slab = Slab(comm.rank, comm.world, n, self.halo)
        self.inner = CudaProgram(chain=chain, device=device, plan_options=plan_options, slab=self.slab)
        self.rt = self.inner.rt
        self.program = self.inner.program
        self.plan = self.inner.plan
        self.lowered = self.inner.lowered
        self.buffers = self.inner.buffers
        self.xplan = ExchangePlan(self.lowered, self.plan.buffer_assignment())
        self.sends = self.xplan.for_rank(self.slab)
        self.comm_streams = {}                 # peer rank -> stream of the copy pushes towards it
        self._push_events = {}                 # (storage id, peer) -> event of the last copy push that read it
        self._launch_events = {}               # launch index [, peer] -> event behind the launch [its copy push]
        self.rep = 0                           # executions so far (the counters never restart)
        self._setup_peers()
        self.inner.push_fn = self._push_params

    # -- forwarding
    def local_shape(self, name):
        return self.inner.local_shape(name)

    @property
    def launch_count(self):
        return self.inner.launch_count

    @property
    def launches_per_execution(self):
        return self.inner.launches_per_execution

    def set_scalars(self, values):
        self.inner.set_scalars(values)

    def input_index_offsets(self):
        """Global flat index of the first allocated element of every slab-decomposed input."""
        offs = {}
        it = "ijk"[self.lowered.slab_axis]
        for name, f in self.program.fields.items():
            if f.kind == "input" and not f.is_scalar and it in f.dims:
                plane = int(np.prod(f.shape[1:])) if f.dims[0] == it else None
                if plane is None:
                    raise ValueError("slab axis must be the outermost dimension of {}".format(name))
                offs[name] = self.slab.alloc_begin * plane
        return offs

    def _plane_elems(self, name):
        f = self.program.fields[name]
        return int(np.prod(f.shape[1:]))

    def _is_sharded(self, name):
        f = self.program.fields[name]
        return (not f.is_scalar) and ("ijk"[self.lowered.slab_axis] in f.dims)

    # -- peers
    F_BELOW, F_ABOVE, P_LOWER, P_UPPER = 0, 4, 8, 12     # byte offsets of the four counters in ``flags``

    def _setup_peers(self):
        rt = self.rt
        # counters other ranks write into this rank's memory: [0] pushes arrived from below (the lower
        # neighbour's "up" channel), [1] from above, [2] progress of the lower neighbour's launches,
        # [3] progress of the upper neighbour's
        self.flags = rt.malloc(256)
        rt.memset(self.flags, 0, 256)
        rt.stream_synchronize()
        storage = {}
        for name, buf in self.buffers.items():
            storage.setdefault(buf.dptr, rt.ipc_get_handle(buf.dptr))
        mine = {"flags": rt.ipc_get_handle(self.flags),
                "buffers": {name: storage[buf.dptr] for name, buf in self.buffers.items()},
                "alloc_begin": self.slab.alloc_begin}
        everyone = self.comm.allgather(pickle.dumps(mine))
        self.peers = {}
        opened = {}
        for peer in (self.comm.rank - 1, self.comm.rank + 1):
            if 0 <= peer < self.comm.world:
                info = pickle.loads(everyone[peer])
                ptrs = {}
                for name, handle in info["buffers"].items():
                    if handle not in opened:
                        opened[handle] = rt.ipc_open_handle(handle)
                    ptrs[name] = opened[handle]
                self.peers[peer] = {"flags": rt.ipc_open_handle(info["flags"]), "buffers": ptrs,
                                    "alloc_begin": info["alloc_begin"]}
                self.comm_streams[peer] = rt.stream_create()
        self._opened = list(opened.values()) + [p["flags"] for p in self.peers.values()]
        self.comm.barrier()

    INT_MIN, INT_MAX = -(2 ** 31), 2 ** 31 - 1

    def _push_params(self, l, field):
        """Kernel arguments of the in-kernel push of ``field`` by launch ``l``: byte distance from this
        rank's buffer to the lower / upper neighbour's (same cell), and the plane thresholds -- planes
        below ``lo_end`` also go down, planes from ``hi_begin`` on also go up."""
        idx = self.lowered.launches.index(l)
        f = self.program.fields[field]
        plane_bytes = self._plane_elems(field) * f.data_type.bytes
        mine = self.buffers[field].dptr
        d_lo = d_hi = 0
        lo_end, hi_begin = self.INT_MIN, self.INT_MAX
        lower, upper = self.peers.get(self.comm.rank - 1), self.peers.get(self.comm.rank + 1)
        for (name, fwd) in self.xplan.down[idx]:
            if name == field and lower is not None:
                d_lo = lower["buffers"][field] - mine + (self.slab.alloc_begin - lower["alloc_begin"]) * plane_bytes
                lo_end = self.slab.begin + fwd
        for (name, back) in self.xplan.up[idx]:
            if name == field and upper is not None:
                d_hi = upper["buffers"][field] - mine + (self.slab.alloc_begin - upper["alloc_begin"]) * plane_bytes
                hi_begin = self.slab.end - back
        return d_lo, d_hi, lo_end, hi_begin

    # -- execution
    def execute(self):
        """All launches of the program on the owned slab.  Fields a later launch reads across the slab
        boundary reach the neighbours' halo planes from inside the producing kernel (streamed passes)
        or by peer copies on the communication streams (one-operator kernels); counters in the
        neighbours' memory order producers, consumers and the reuse of halo storage (``ExchangePlan``)."""
        inner, rt, x = self.inner, self.rt, self.xplan
        if inner._packs is None:
            inner._build_packs()
        stream = rt.stream
        rank = self.comm.rank
        rep = self.rep
        self.rep += 1
        lower, upper = self.peers.get(rank - 1), self.peers.get(rank + 1)
        flags = self.flags
        assign = self.plan.buffer_assignment()
        by_launch: Dict[int, List[HaloSend]] = {}
        for s in self.sends:
            by_launch.setdefault(s.launch, []).append(s)
        for idx, (l, fn, grid, pack) in enumerate(inner._packs):
            # read-after-write: the halos this launch reads must have arrived
            need_lo, need_hi = x.wait_values(rep, idx)
            if lower is not None and need_lo:
                rt.wait_flag(stream, flags + self.F_BELOW, need_lo)
            if upper is not None and need_hi:
                rt.wait_flag(stream, flags + self.F_ABOVE, need_hi)
            sends = by_launch.get(idx, [])
            in_kernel = bool(l.info.get("peer_push")) and bool(sends)
            war = x.war_value(rep, idx)
            if in_kernel and war:
                # the kernel itself writes into the neighbours' halo planes: their last readers must be done
                for peer in sorted({s.peer for s in sends}):
                    rt.wait_flag(stream, flags + (self.P_LOWER if peer < rank else self.P_UPPER), war)
            # a copy push of an earlier launch may still be reading storage this launch overwrites
            for f in l.writes:
                for peer in self.peers:
                    ev = self._push_events.pop((assign.get(f, f), peer), None)
                    if ev is not None:
                        rt.stream_wait_event(stream, ev)
            rt.launch(fn, grid, l.block, l.smem, pack.array, stream)
            if in_kernel:
                if x.up[idx] and upper is not None:
                    rt.write_flag(stream, upper["flags"] + self.F_BELOW, x.arrival_value("up", rep, idx))
                if x.down[idx] and lower is not None:
                    rt.write_flag(stream, lower["flags"] + self.F_ABOVE, x.arrival_value("down", rep, idx))
            elif sends:
                ev = self._launch_events.get(idx)
                if ev is None:
                    ev = self._launch_events[idx] = rt.event_create(False)
                rt.event_record(ev, stream)
                for peer in sorted({s.peer for s in sends}):
                    cs = self.comm_streams[peer]
                    rt.stream_wait_event(cs, ev)
                    if war:
                        rt.wait_flag(cs, flags + (self.P_LOWER if peer < rank else self.P_UPPER), war)
                    for s in sends:
                        if s.peer != peer:
                            continue
                        f = self.program.fields[s.field]
                        plane_bytes = self._plane_elems(s.field) * f.data_type.bytes
                        info = self.peers[peer]
                        src = self.buffers[s.field].dptr + (s.src_begin - self.slab.alloc_begin) * plane_bytes
                        dst = info["buffers"][s.field] + (s.src_begin - info["alloc_begin"]) * plane_bytes
                        rt.d2d(dst, src, (s.src_end - s.src_begin) * plane_bytes, cs)
                    if peer > rank:
                        rt.write_flag(cs, info["flags"] + self.F_BELOW, x.arrival_value("up", rep, idx))
                    else:
                        rt.write_flag(cs, info["flags"] + self.F_ABOVE, x.arrival_value("down", rep, idx))
                    done = self._launch_events.get((idx, peer))
                    if done is None:
                        done = self._launch_events[(idx, peer)] = rt.event_create(False)
                    rt.event_record(done, cs)
                    for s in sends:
                        if s.peer == peer:
                            self._push_events[(assign.get(s.field, s.field), peer)] = done
            if idx in x.progress_points:
                value = rep * x.n + idx + 1
                if lower is not None:
                    rt.write_flag(stream, lower["flags"] + self.P_UPPER, value)     # I am their upper neighbour
                if upper is not None:
                    rt.write_flag(stream, upper["flags"] + self.P_LOWER, value)     # I am their lower neighbour
        inner.launch_count += len(inner._packs)

    # -- the reference-facing call with host arrays
    def __call__(self, **kwargs):
        """Run once with this rank's planes as host arrays (``local_shape``: owned planes + halo):
        inputs are copied in, the program runs, owned output planes are copied back in place.  When
        the buffers carry the accumulated reach of the program the call is cut into pieces whose
        copies and passes overlap and needs no halo exchange at all (``CudaProgram._pipeline_schedule``);
        otherwise: copy in, ``execute()`` with NVLink halo pushes, copy out."""
        inner, rt = self.inner, self.rt
        arrays, scalars = inner._split_call_args(kwargs)
        if scalars:
            inner.set_scalars(scalars)
        pieces = int(os.environ.get("SFB200_PIPELINE_PIECES", "16"))
        fields = self.program.fields
        in_out = [n for n, f in fields.items() if not f.is_scalar and f.kind in ("input", "output")]
        if pieces > 1 and all(n in arrays for n in in_out) and inner._call_pipelined(arrays, pieces):
            self.last_call_bytes = inner.last_call_bytes
            return
        h2d = d2h = 0
        for name, f in fields.items():
            if f.kind == "input" and not f.is_scalar:
                if name not in arrays:
                    raise KeyError("input array {} was not provided".format(name))
                n = int(np.prod(self.local_shape(name)))
                arr = np.ascontiguousarray(np.asarray(arrays[name], dtype=f.data_type.type)).reshape(-1)
                if arr.size < n:
                    raise ValueError("input {} has {} elements, this rank's slab needs {}".format(name, arr.size, n))
                rt.h2d(self.buffers[name].dptr, arr[:n])
                h2d += n * f.data_type.bytes
        self.execute()
        for name in self.program.outputs:
            if name not in arrays:
                continue
            f = fields[name]
            out = np.asarray(arrays[name])
            n = int(np.prod(self.local_shape(name)))
            if out.size != n or out.dtype != f.data_type.type or not out.flags["C_CONTIGUOUS"]:
                raise ValueError("output array for {} must be C-contiguous {} of {} elements".format(
                    name, f.data_type, n))
            flat = out.reshape(-1)
            # owned planes only: the halo planes of the device buffer hold the neighbours' data
            if self._is_sharded(name):
                plane = self._plane_elems(name)
                lo = (self.slab.begin - self.slab.alloc_begin) * plane
                hi = (self.slab.end - self.slab.alloc_begin) * plane
            else:
                lo, hi = 0, n
            rt.d2h(flat[lo:hi], self.buffers[name].dptr + lo * f.data_type.bytes)
            d2h += (hi - lo) * f.data_type.bytes
        rt.stream_synchronize()
        self.last_call_bytes = (h2d, d2h)

    # -- host data movement (parity runs; the benchmark generates its fields in HBM)
    def upload_global(self, name, array):
        """Copy this rank's allocated planes of a *global* host array to the device."""
        f = self.program.fields[name]
        arr = np.ascontiguousarray(np.asarray(array, dtype=f.data_type.type).reshape(f.shape))
        if self._is_sharded(name):
            arr = np.ascontiguousarray(arr[self.slab.alloc_begin:self.slab.alloc_end])
        self.rt.h2d(self.buffers[name].dptr, arr)
        self.rt.stream_synchronize()

    def download_owned(self, name):
        """Owned planes of a field as a host array."""
        local = self.inner.download(name)
        if not self._is_sharded(name):
            return local
        lo = self.slab.begin - self.slab.alloc_begin
        return np.ascontiguousarray(local[lo:lo + (self.slab.end - self.slab.begin)])

    def gather(self, name):
        """Full field on every rank (parity checks at reduced size only)."""
        parts = self.comm.allgather(self.download_owned(name))
        return np.concatenate(parts, axis=0) if self._is_sharded(name) else parts[0]

    def checksum_owned(self, name):
        """(sum, bit checksum) of the owned planes, computed on the device."""
        f = self.program.fields[name]
        plane = self._plane_elems(name)
        lo = (self.slab.begin - self.slab.alloc_begin) * plane if self._is_sharded(name) else 0
        n = (self.slab.end - self.slab.begin) * plane if self._is_sharded(name) else f.size
        return self.rt.checksum(self.buffers[name].dptr + lo * f.data_type.bytes, n, f.data_type.type)

    def close(self):
        self.rt.stream_synchronize()
        self.comm.barrier()
        for p in self._opened:
            try:
                self.rt.ipc_close_handle(p)
            except Exception:
                pass
        for ev in self._launch_events.values():
            self.rt.event_destroy(ev)
        self._launch_events, self._push_events = {}, {}
        self.rt.free(self.flags)
        self.inner.close()
