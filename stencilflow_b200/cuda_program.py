"""The compiled program object of ``cuda`` mode.

``CudaProgram`` plays the role of the ``CompiledSDFG`` that ``sdfg.compile()`` hands to the reference
driver (``stencilflow/run_program.py:123,164-172``; ``dace/dace/codegen/compiled_sdfg.py:269-294``):
it is called with keyword arguments ``<input>_host=ndarray``, ``<scalar>=value`` and
``<output>_host=ndarray`` (un-suffixed names are accepted too, as the reference's CPU program takes
them, ``run_program.py:186-192``); outputs are caller-allocated and written in place.

Underneath: front end -> operator 5-tuples -> planner -> generated sm_100a CUDA C++ -> NVRTC cubin
(cached under ``.sfcache/``) -> module -> launches on one stream, all through ``libsfb200.so``.
"""

import ctypes
import hashlib
import json
import os
import time

import numpy as np

from . import planner as _planner
from . import runtime as rt
from .kernel_chain_graph import KernelChainGraph
from .log_level import LogLevel
from .stencil_op import make_program

NVRTC_OPTIONS = ["-arch=sm_100a", "-std=c++17", "-lineinfo", "--use_fast_math=false"]

_REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cache_root():
    return os.environ.get("SFB200_CACHE", os.path.join(_REPO_ROOT, ".sfcache"))


def compile_cached(name, source, options=None):
    """Generated CUDA C++ -> cubin bytes, cached on disk by content hash (the counterpart of
    ``.dacecache/<name>/`` and ``-use-cached-sdfg``, ``stencilflow/run_program.py:69-73``).
    Returns (cubin, directory, was_cached)."""
    options = [o for o in (options or NVRTC_OPTIONS) if o != "--use_fast_math=false"]
    key = hashlib.sha1((source + "\0" + " ".join(options)).encode()).hexdigest()[:16]
    directory = os.path.join(cache_root(), "{}-{}".format(name, key))
    cubin_path = os.path.join(directory, "kernel.cubin")
    src_path = os.path.join(directory, "kernel.cu")
    if os.path.isfile(cubin_path) and os.path.isfile(src_path):
        with open(cubin_path, "rb") as f:
            return f.read(), directory, True
    os.makedirs(directory, exist_ok=True)
    with open(src_path, "w") as f:
        f.write(source)
    image, log = rt.compile_source(source, src_path, options)
    tmp = cubin_path + ".tmp{}".format(os.getpid())
    with open(tmp, "wb") as f:
        f.write(image)
    os.replace(tmp, cubin_path)
    if log.strip():
        with open(os.path.join(directory, "nvrtc.log"), "w") as f:
            f.write(log)
    return image, directory, False


class DeviceBuffer:
    def __init__(self, name, nbytes, dptr):
        self.name = name
        self.nbytes = nbytes
        self.dptr = dptr


class CudaProgram:
    def __init__(self, stencil_file=None, chain=None, log_level=LogLevel.NO_LOG, device=None,
                 plan_options=None, specialize_scalars=None, synthetic_reads=None,
                 allocate=True, slab=None):
        """``slab``: None for a whole-domain program, or a :class:`distributed.Slab` describing the
        part of the outermost dimension this process owns (multi-GPU)."""
        if chain is None:
            chain = KernelChainGraph(stencil_file, log_level=log_level)
        self.chain = chain
        self.name = chain.name.replace(".", "_")
        self.program = make_program(chain)
        self.slab = slab
        self.synthetic_reads = synthetic_reads
        self.plan = _planner.plan_program(self.program, options=plan_options,
                                          specialize=specialize_scalars)
        self.lowered = self.plan.lowered
        self.image, self.cache_dir, self.was_cached = compile_cached(self.name, self.lowered.source)
        with open(os.path.join(self.cache_dir, "plan.json"), "w") as f:
            json.dump(self.plan.describe(), f, indent=1)
        self.rt = None
        self.handle = None
        self.module = None
        self.functions = {}
        self.buffers = {}          # field -> DeviceBuffer
        self._owned = []
        self._tables = []          # work tables of persistent launches (device memory)
        self._packs = None
        self._graph = None
        self._capturing = False
        self.scalar_values = {}
        self.launch_count = 0
        if allocate:
            self.load(device)

    # ------------------------------------------------------------------ device set-up
    def load(self, device=None):
        self.rt = rt.Runtime.get(device)
        self.module = self.rt.module_load(self.image)
        for name, k in self.lowered.kernels.items():
            fn = self.rt.get_function(self.module, name)
            self.functions[name] = fn
        for l in self.lowered.launches:
            if l.smem > 48 * 1024:
                self.rt.set_max_dynamic_smem(self.functions[l.kernel], l.smem)
        # the per-program handle of the C ABI (whole-domain programs; a slab's launches depend on its neighbours)
        self.handle = self.rt.program_create(self.image) if self.slab is None else None
        self._handle_index = {}
        self._allocate()

    def local_shape(self, field):
        """Shape of a field's device buffer (slab extent + halos along the slab axis)."""
        f = self.program.fields[field]
        if self.slab is None or self.lowered.slab_axis is None:
            return f.shape
        it = "ijk"[self.lowered.slab_axis]
        if it not in f.dims:
            return f.shape
        shape = list(f.shape)
        shape[f.dims.index(it)] = self.slab.alloc_end - self.slab.alloc_begin
        return tuple(shape)

    def _allocate(self):
        fields = self.program.fields
        assign = self.plan.buffer_assignment()        # materialised field -> storage id
        storage = {}
        for name, sid in assign.items():
            f = fields[name]
            nbytes = int(np.prod(self.local_shape(name))) * f.data_type.bytes
            storage[sid] = max(storage.get(sid, 0), nbytes)
        ptrs = {}
        if self.handle is not None:
            # whole-domain program: the library's program handle owns the fields (sfb_program_add_buffer)
            first = {}
            for name, sid in assign.items():
                if sid not in first:
                    first[sid] = self.rt.program_add_buffer(self.handle, name, storage[sid])
                    self._handle_index[name] = first[sid]
                else:
                    self._handle_index[name] = self.rt.program_add_buffer(self.handle, name, storage[sid], first[sid])
                ptrs[sid] = self.rt.program_buffer(self.handle, name)[0]
        else:
            for sid, nbytes in storage.items():
                ptrs[sid] = self.rt.malloc(nbytes)
                self._owned.append(ptrs[sid])
        for name, sid in assign.items():
            self.buffers[name] = DeviceBuffer(name, storage[sid], ptrs[sid])
        self.device_bytes = sum(storage.values())

    def close(self):
        if self.rt is None:
            return
        self._unpin_all()
        if self._graph is not None:
            self.rt.graph_destroy(self._graph)
            self._graph = None
        for p in self._owned + self._tables:
            self.rt.free(p)
        self._owned, self._tables = [], []
        self.buffers = {}
        if getattr(self, "handle", None) is not None:
            self.rt.program_destroy(self.handle)
            self.handle = None
        if self.module is not None:
            self.rt.module_unload(self.module)
            self.module = None

    # ------------------------------------------------------------------ execution
    def _slab_range(self):
        axis = self.lowered.slab_axis
        if axis is None:
            return 0, 0, 1
        n = self.program.shape3[axis]
        if self.slab is None:
            return 0, 0, n
        return self.slab.alloc_begin, self.slab.begin, self.slab.end

    def set_scalars(self, values):
        for k, v in values.items():
            self.scalar_values[k] = v
        self._packs = None
        if self._graph is not None:
            self.rt.graph_destroy(self._graph)
            self._graph = None

    def _build_packs(self):
        s_base, s_begin, s_end = self._slab_range()
        self._packs = [self._pack_launch(l, s_base, s_begin, s_end, push=True) for l in self.lowered.launches]
        if self.handle is not None:
            # one library call then runs the whole program: the handle keeps every launch with its parameters
            self.rt.program_clear_launches(self.handle)
            for l, fn, grid, pack in self._packs:
                self._handle_add_launch(l, grid, pack.specs)

    def _pack_launch(self, l, s_base, s_begin, s_end, push=False):
        """(launch, function, grid, parameter pack) of launch ``l`` producing planes
        [s_begin, s_end) of the slab axis, device buffers starting at plane ``s_base``.  ``push``: let a
        slab kernel store its edge planes into the neighbouring GPUs' halos (``SlabProgram.execute``
        only; ``push_fn`` is installed by the slab program)."""
        b0, e0 = l.info.get("range_fn", lambda b, e: (b, e))(s_begin, s_end)
        specs = self._param_specs(l, s_base, b0, e0, push)
        vals = []
        for spec in specs:
            if spec[0] == "bytes":
                vals.append(spec[1])
            elif spec[0] == "buffer":
                vals.append(ctypes.c_void_p(self.buffers[spec[1]].dptr))
            elif spec[0] == "tmap":
                _, field, dt, dims, strides, box = spec
                vals.append(self.rt.tensor_map(self.buffers[field].dptr, dt, dims, strides, box))
            elif spec[0] == "table":
                dptr = self.rt.malloc(spec[1].nbytes)
                self._tables.append(dptr)
                self.rt.h2d(dptr, spec[1])
                self.rt.stream_synchronize()
                vals.append(ctypes.c_void_p(dptr))
        pack = rt.pack_params(vals)
        pack.specs = specs
        return (l, self.functions[l.kernel], self._grid(l, b0, e0), pack)

    def _grid(self, l, b0, e0):
        if l.info.get("persistent"):
            return l.grid_fn(b0, e0, self._resident_ctas(l))
        return l.grid_fn(b0, e0)

    def _param_specs(self, l, s_base, b0, e0, push=False):
        """The parameters of launch ``l`` for planes [b0, e0), independent of who launches it:
        ``("bytes", ctypes value)`` | ``("buffer", field)`` | ``("tmap", field, dtype, dims, strides, box)``
        | ``("table", int32 array)``."""
        specs = []
        for a in l.args:
            if a[0] == "buf":
                specs.append(("buffer", a[1]))
            elif a[0] == "scalar":
                dt, name = a[1], a[2]
                if name not in self.scalar_values:
                    raise KeyError("scalar input {} was not provided".format(name))
                specs.append(("bytes", np.ctypeslib.as_ctypes_type(dt.type)(self.scalar_values[name])))
            elif a[0] == "slab":
                specs += [("bytes", ctypes.c_int(s_base)), ("bytes", ctypes.c_int(b0)), ("bytes", ctypes.c_int(e0))]
            elif a[0] == "int":
                specs.append(("bytes", ctypes.c_int(a[1])))
            elif a[0] == "chunk":
                specs.append(("bytes", ctypes.c_int(l.info["chunk_fn"](b0, e0))))
            elif a[0] == "push":
                fn_ = getattr(self, "push_fn", None) if push else None
                d_lo, d_hi, lo_end, hi_begin = fn_(l, a[1]) if fn_ else (0, 0, -(2 ** 31), 2 ** 31 - 1)
                specs += [("bytes", ctypes.c_longlong(d_lo)), ("bytes", ctypes.c_longlong(d_hi)),
                          ("bytes", ctypes.c_int(lo_end)), ("bytes", ctypes.c_int(hi_begin))]
            elif a[0] == "worktab":
                specs.append(("table", np.ascontiguousarray(
                    np.asarray(l.info["work_fn"](b0, e0, self._resident_ctas(l)), dtype=np.int32))))
            elif a[0] == "tmap":
                spec = a[1]
                shape = self.local_shape(spec["field"])
                dt = self.program.fields[spec["field"]].data_type
                dims = list(reversed(shape))
                strides = []
                acc = dt.bytes
                for d in dims[:-1]:
                    acc *= d
                    strides.append(acc)
                specs.append(("tmap", spec["field"], dt, dims, strides, list(spec["box"])))
            else:
                raise ValueError(a)
        return specs

    def _handle_add_launch(self, l, grid, specs):
        """The same launch described to the library's program handle (``sfb_program_add_launch``)."""
        params, keep = [], []
        for spec in specs:
            q = rt.LaunchParam()
            if spec[0] == "bytes":
                q.kind, q.size = rt.PARAM_BYTES, ctypes.sizeof(spec[1])
                q.data = ctypes.addressof(spec[1])
                keep.append(spec[1])
            elif spec[0] == "buffer":
                q.kind, q.buffer = rt.PARAM_BUFFER, self._handle_index[spec[1]]
            elif spec[0] == "tmap":
                _, field, dt, dims, strides, box = spec
                q.kind, q.buffer = rt.PARAM_TMAP, self._handle_index[field]
                q.dtype, q.rank = rt.dtype_code(dt), len(dims)
                for k, d in enumerate(dims):
                    q.dims[k] = d
                    q.box[k] = box[k]
                for k, st in enumerate(strides):
                    q.strides_bytes[k] = st
            elif spec[0] == "table":
                q.kind, q.size = rt.PARAM_TABLE, spec[1].nbytes
                q.data = spec[1].ctypes.data
                keep.append(spec[1])
            params.append(q)
        self.rt.program_add_launch(self.handle, l.kernel, grid, l.block, l.smem, params, keep)

    def export_plan(self, directory, inputs=None):
        """Writes what a host in another language needs to run this program through the per-program
        handle of the C ABI (``sfb_program_*``): ``kernel.cubin``, ``program.sfbplan`` (fields, launches
        with their parameters, input/output files) and, if ``inputs`` are given, the raw ``.dat`` input
        arrays.  ``examples/run_sfbplan.c`` is such a host.  Needs a device (the grids of persistent
        kernels depend on its occupancy).  Returns the path of the plan script."""
        if self.slab is not None:
            raise ValueError("a slab program is driven by its rank, not by a plan script")
        if inputs:
            self.set_scalars({k: v for k, v in inputs.items() if self.program.fields[k].is_scalar})
        if self._packs is None:
            self._build_packs()
        os.makedirs(directory, exist_ok=True)
        with open(os.path.join(directory, "kernel.cubin"), "wb") as f:
            f.write(self.image)
        names = list(self._handle_index)
        order = sorted(names, key=lambda n: self._handle_index[n])
        assign = self.plan.buffer_assignment()
        first = {}
        lines = ["image {}".format(os.path.join(directory, "kernel.cubin"))]
        for name in order:
            sid = assign[name]
            share = first.get(sid, -1)
            first.setdefault(sid, self._handle_index[name])
            lines.append("buffer {} {} {}".format(name, self.buffers[name].nbytes, share))
        for l, fn, grid, pack in self._packs:
            lines.append("launch {} {} {} {} {} {} {} {} {}".format(l.kernel, *grid, *l.block, l.smem, len(pack.specs)))
            for spec in pack.specs:
                if spec[0] == "bytes":
                    raw = bytes(spec[1])
                    lines.append("  bytes {} {}".format(len(raw), raw.hex()))
                elif spec[0] == "buffer":
                    lines.append("  buffer {} 0".format(self._handle_index[spec[1]]))
                elif spec[0] == "tmap":
                    _, field, dt, dims, strides, box = spec
                    lines.append("  tmap {} {} {} {}".format(self._handle_index[field], rt.dtype_code(dt), len(dims),
                                                             " ".join(map(str, list(dims) + list(strides) + list(box)))))
                elif spec[0] == "table":
                    lines.append("  table {} {}".format(spec[1].size, " ".join(map(str, spec[1].tolist()))))
        for name, f in self.program.fields.items():
            if f.is_scalar or f.kind == "intermediate":
                continue
            path = os.path.join(directory, name + ".dat")
            if f.kind == "input":
                if inputs is not None and name in inputs:
                    np.ascontiguousarray(np.asarray(inputs[name], dtype=f.data_type.type)).tofile(path)
                lines.append("input {} {}".format(name, path))
            else:
                lines.append("output {} {}".format(name, path))
        script = os.path.join(directory, "program.sfbplan")
        with open(script, "w") as f:
            f.write("\n".join(lines) + "\n")
        return script

    def _resident_ctas(self, l):
        """CTA slots of the device for a persistent streamed kernel: SMs x the occupancy the driver
        reports for the loaded function (one CTA per slot streams an equal share of the pass)."""
        cache = self.__dict__.setdefault("_slots", {})
        if l.kernel not in cache:
            per_sm = self.rt.occupancy(self.functions[l.kernel], l.block[0], l.smem)
            if per_sm < 1:
                raise rt.SfbError(-1, "kernel {} does not fit an SM ({} threads, {} bytes of shared memory)".format(
                    l.kernel, l.block[0], l.smem))
            cache[l.kernel] = per_sm * int(self.rt.props.sm_count)
        return cache[l.kernel]

    GRAPH_MAX_CELLS = 1 << 21

    def execute(self, stream=None):
        """Enqueue every launch of the plan (asynchronous).  Launch-bound programs -- several launches
        over a grid so small that each kernel runs for a few microseconds -- go through a captured CUDA
        graph, which takes the per-launch driver work off the critical path (``SFB200_GRAPH=0``: never)."""
        if self._packs is None:
            self._build_packs()
        if (stream is None and not self._capturing and self.slab is None and len(self._packs) >= 3
                and self.program.cells <= self.GRAPH_MAX_CELLS and os.environ.get("SFB200_GRAPH", "1") != "0"):
            return self.execute_graph()
        if self.handle is not None:
            self.rt.program_run(self.handle, 1, stream)          # all launches in one library call
        else:
            for l, fn, grid, pack in self._packs:
                self.rt.launch(fn, grid, l.block, l.smem, pack.array, stream)
        self.launch_count += len(self._packs)

    def execute_graph(self):
        """Same as :meth:`execute` through a captured CUDA graph (launch-bound programs)."""
        if self._packs is None:
            self._build_packs()
        if self._graph is None:
            self.rt.graph_begin()
            self._capturing = True
            try:
                self.execute()
            finally:
                self._capturing = False
                self._graph = self.rt.graph_end()
        else:
            self.launch_count += len(self._packs)
        self.rt.graph_launch(self._graph)

    @property
    def launches_per_execution(self):
        return len(self.lowered.launches)

    def upload(self, name, array):
        f = self.program.fields[name]
        shape = self.local_shape(name)
        n = int(np.prod(shape))
        arr = np.asarray(array)
        if arr.dtype != f.data_type.type:
            arr = arr.astype(f.data_type.type)
        if arr.size < n:
            raise ValueError("input {} has {} elements, the program needs {}".format(name, arr.size, n))
        if arr.shape != tuple(shape):
            # the reference hands lower-dimensional inputs over at the full program shape and embedded
            # lists flat; the program reads the first prod(shape) elements (helper.py:162-217)
            arr = np.ascontiguousarray(arr).ravel()[:n]
        arr = np.ascontiguousarray(arr)
        self.rt.h2d(self.buffers[name].dptr, arr, nbytes=n * f.data_type.bytes)
        self.rt.stream_synchronize()

    def download(self, name, out=None):
        f = self.program.fields[name]
        shape = self.local_shape(name)
        if out is None:
            out = np.empty(shape, dtype=f.data_type.type)
        n = int(np.prod(shape))
        if out.size != n or out.dtype != f.data_type.type or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("output array for {} must be C-contiguous {} of {} elements".format(
                name, f.data_type, n))
        self.rt.d2h(out, self.buffers[name].dptr, nbytes=n * f.data_type.bytes)
        self.rt.stream_synchronize()
        return out

    def _split_call_args(self, kwargs):
        arrays, scalars = {}, {}
        for key, val in kwargs.items():
            name = key[:-5] if key.endswith("_host") and key[:-5] in self.program.fields else key
            if name not in self.program.fields:
                raise KeyError("unknown program argument {}".format(key))
            if self.program.fields[name].is_scalar:
                scalars[name] = val
            else:
                arrays[name] = val
        return arrays, scalars

    # ------------------------------------------------------------------ pipelined host call
    PIPELINE_MIN_BYTES = 64 << 20

    def _pipeline_schedule(self, pieces):
        """:meth:`_pipeline_ranges` with every launch range turned into a parameter pack."""
        ranges = self._pipeline_ranges(pieces)
        if ranges is None:
            return None
        base = self.slab.alloc_begin if self.slab is not None else 0
        for step in ranges:
            step["launch"] = [self._pack_launch(self.lowered.launches[idx], base, b, e)
                              for (idx, b, e) in step["launch"]]
        return ranges

    def _pipeline_ranges(self, pieces):
        """Cuts one execution into ``pieces`` along the slab axis so that host->device copies, the
        passes and device->host copies of different pieces overlap (PCIe is full duplex).

        Piece s makes input planes < e_s available; every launch then advances as far as the planes
        it reads allow (its output frontier trails its inputs' by its forward reach), so nothing is
        computed twice and no launch reads a plane that is not final.

        On a slab (one rank of a multi-GPU run) the same schedule runs on the rank's own planes without
        any halo exchange: launch l produces the owned range widened by what the launches after it
        still reach for (those planes are recomputed redundantly on both neighbours, bit-identically),
        which needs the buffers to carry the *accumulated* reach of the program as halo
        (``distributed.total_reach``).

        Returns a list of steps ``{"h2d": [(field, b, e)], "launch": [(launch index, b, e)], "d2h":
        [(field, b, e)]}`` (plane ranges along the slab axis, global numbering), or None when the plan
        cannot be cut: no slab axis, a cluster plan (one launch computes the whole program), an array that does not span it,
        intermediates that share storage (a later piece would still need planes an earlier piece's
        successor overwrote), or a slab whose halo is thinner than the accumulated reach."""
        lowered = self.lowered
        axis = lowered.slab_axis
        if axis is None or pieces < 2 or any(l.family == "cluster" for l in lowered.launches):
            return None
        it = "ijk"[axis]
        fields = self.program.fields
        n = self.program.shape3[axis]
        arrays = [name for name, f in fields.items() if not f.is_scalar and f.kind in ("input", "output")]
        # inputs without the slab axis (1-D/2-D coefficient arrays) are small: they go up whole with
        # the first piece; everything else must have the slab axis outermost
        whole = [a for a in arrays if fields[a].kind == "input" and it not in fields[a].dims]
        arrays = [a for a in arrays if a not in whole]
        if any(it not in fields[a].dims or fields[a].dims[0] != it for a in arrays):
            return None
        assign = self.plan.buffer_assignment()
        if len(set(assign.values())) != len(assign):
            return None
        if self.slab is None:
            dom0, dom1, own0, own1 = 0, n, 0, n
        else:
            dom0, dom1, own0, own1 = self.slab.alloc_begin, self.slab.alloc_end, self.slab.begin, self.slab.end
        from .distributed import launch_reach
        launches = lowered.launches
        reach = [launch_reach(lowered, idx) for idx in range(len(launches))]
        if (dom1 - dom0) // pieces < 4 * max([1] + [max(r) for rr in reach for r in rr.values()]):
            return None
        inputs = [a for a in arrays if fields[a].kind == "input"]
        outputs = [a for a in arrays if fields[a].kind == "output"]
        # planes every launch has to produce, and planes of every field somebody needs
        need = {o: [own0, own1] for o in outputs}
        target = [None] * len(launches)
        for idx in range(len(launches) - 1, -1, -1):
            l = launches[idx]
            wanted = [need[w] for w in l.writes if w in need]
            if not wanted:
                return None
            lo, hi = min(w[0] for w in wanted), max(w[1] for w in wanted)
            target[idx] = (lo, hi)
            for f in l.reads:
                if fields[f].is_scalar or it not in fields[f].dims:
                    continue
                b, fw = reach[idx].get(f, (0, 0))
                r = need.setdefault(f, [n, 0])
                r[0], r[1] = min(r[0], max(0, lo - b)), max(r[1], min(n, hi + fw))
        for a in inputs:
            need.setdefault(a, [own0, own1])
            if need[a][0] < dom0 or need[a][1] > dom1:
                return None
        avail = {a: need[a][0] for a in inputs}
        top = {a: need[a][1] for a in inputs}
        for idx, l in enumerate(launches):
            for f in l.writes:
                top[f] = target[idx][1]
        done = [t[0] for t in target]
        out_done = {o: own0 for o in outputs}
        span0 = min(need[a][0] for a in inputs)
        span1 = max(need[a][1] for a in inputs)
        schedule = []
        max_reach = max([1] + [max(r) for rr in reach for r in rr.values()])
        for s, e_in in enumerate(self._piece_ends(span0, span1, pieces, max_reach)):
            step = {"h2d": [], "launch": [], "d2h": [], "h2d_whole": whole if s == 0 else []}
            for a in inputs:
                e_a = min(max(e_in, avail[a]), need[a][1])
                step["h2d"].append((a, avail[a], e_a))
                avail[a] = e_a
            for idx, l in enumerate(launches):
                lim = target[idx][1]
                for f in l.reads:
                    if f not in avail:
                        continue
                    have = avail[f]
                    fwd = reach[idx].get(f, (0, 0))[1]
                    lim = min(lim, target[idx][1] if have >= top[f] else have - fwd)
                lim = max(lim, done[idx])
                if lim > done[idx]:
                    step["launch"].append((idx, done[idx], lim))
                    done[idx] = lim
                for f in l.writes:
                    avail[f] = lim
            for o in outputs:
                e_o = min(avail.get(o, own0), own1)
                if e_o > out_done[o]:
                    step["d2h"].append((o, out_done[o], e_o))
                    out_done[o] = e_o
            schedule.append(step)
        assert all(d == t[1] for d, t in zip(done, target)) and all(v == own1 for v in out_done.values())
        return schedule

    @staticmethod
    def _piece_ends(span0, span1, pieces, max_reach):
        """End planes of the pieces of a pipelined call.  The call costs the longer copy direction plus what
        cannot overlap: the upload of the first piece and the download of the last.  So the pieces at both
        ends are short -- 4 x the largest reach, doubling towards the uniform size in the middle -- and only the
        middle of the domain is cut evenly (``SFB200_PIPELINE_RAMP=0``: all pieces equal)."""
        n = span1 - span0
        uniform = [span0 + (n * (s + 1)) // pieces for s in range(pieces)]
        if os.environ.get("SFB200_PIPELINE_RAMP", "1") == "0":
            return uniform
        base = n // pieces
        head, size = [], max(4 * max_reach, 8)
        while size < base:
            head.append(size)
            size *= 2
        if not head or 2 * sum(head) + base > n:
            return uniform
        middle = n - 2 * sum(head)
        k = max(1, int(round(middle / float(base))))
        sizes = head + [middle // k + (1 if q < middle % k else 0) for q in range(k)] + head[::-1]
        ends, pos = [], span0
        for sz in sizes:
            pos += sz
            ends.append(pos)
        assert ends[-1] == span1
        return ends

    # ------------------------------------------------------------------ caller-owned host arrays
    REGISTER_MIN_BYTES = 32 << 20

    def _pin(self, arr):
        """Page-locks a large caller-owned array (``cudaHostRegister`` through ``sfb_host_register``) so
        that its copies are asynchronous DMA at full PCIe rate instead of staged through the driver's
        bounce buffer -- what makes the overlapped call work for the plain numpy arrays the reference
        driver allocates (``stencilflow/run_program.py:145-159``), not only for ``sfb_host_alloc`` memory.
        Registered once per allocation (cached by address), released when the array dies or the
        program is closed.  Failure to register is not an error: the copies are merely slower."""
        import weakref
        base = arr
        while isinstance(getattr(base, "base", None), np.ndarray):
            base = base.base
        if base.nbytes < self.REGISTER_MIN_BYTES or not base.flags["C_CONTIGUOUS"]:
            return False
        pinned = self.__dict__.setdefault("_pinned", {})
        key = (base.ctypes.data, base.nbytes)
        if key in pinned:
            return True
        try:
            if not self.rt.host_register(base):
                pinned[key] = None             # page-locked already (sfb_host_alloc memory, another program)
                return True
        except rt.SfbError:
            pinned[key] = None
            return False
        addr, rtm = base.ctypes.data, self.rt

        def release(addr=addr, key=key, pinned=pinned, rtm=rtm):
            if pinned.pop(key, None) is not None:
                try:
                    rtm.lib.sfb_host_unregister(ctypes.c_void_p(addr))
                except Exception:
                    pass

        try:
            pinned[key] = weakref.finalize(base, release)
        except TypeError:                      # not weak-referenceable: keep it registered until close()
            pinned[key] = release
        return True

    def _unpin_all(self):
        for key, fin in list(self.__dict__.get("_pinned", {}).items()):
            if fin is not None:
                fin()
        self.__dict__["_pinned"] = {}

    def _call_pipelined(self, arrays, pieces):
        key = ("pipeline", pieces)
        if getattr(self, "_pipe_key", None) != key or self._packs is None:
            if self._packs is None:
                self._build_packs()
            self._pipe = self._pipeline_schedule(pieces)
            self._pipe_key = key
            if self._pipe is not None:
                if not hasattr(self, "_pipe_streams"):
                    self._pipe_streams = (self.rt.stream_create(), self.rt.stream_create())
                    self._pipe_events = []
                while len(self._pipe_events) < len(self._pipe):      # one pair per piece (pieces may be ramped)
                    self._pipe_events.append((self.rt.event_create(False), self.rt.event_create(False)))
        if self._pipe is None:
            return False
        rtm, fields = self.rt, self.program.fields
        s_in, s_out = self._pipe_streams
        flat = {}
        for name, arr in arrays.items():
            f = fields[name]
            arr = np.asarray(arr)
            if (arr.dtype != f.data_type.type or not arr.flags["C_CONTIGUOUS"]
                    or arr.size != int(np.prod(self.local_shape(name)))):
                return False
            flat[name] = arr.reshape(-1)
            self._pin(arr)
        base = self.slab.alloc_begin if self.slab is not None else 0     # first plane the buffers hold
        copied = [0, 0]
        start = rtm.event_create(False)
        rtm.event_record(start)                    # copies must not overtake earlier work on the main stream
        rtm.stream_wait_event(s_in, start)
        rtm.stream_wait_event(s_out, start)
        for step, (ev_in, ev_done) in zip(self._pipe, self._pipe_events):
            for name in step.get("h2d_whole", ()):
                rtm.h2d(self.buffers[name].dptr, flat[name], stream=s_in)
                copied[0] += flat[name].nbytes
            for (name, b, e) in step["h2d"]:
                f = fields[name]
                plane = int(np.prod(f.shape[1:])) if len(f.shape) > 1 else 1
                if e > b:
                    rtm.h2d(self.buffers[name].dptr + (b - base) * plane * f.data_type.bytes,
                            flat[name][(b - base) * plane:(e - base) * plane], stream=s_in)
                    copied[0] += (e - b) * plane * f.data_type.bytes
            rtm.event_record(ev_in, s_in)
            rtm.stream_wait_event(None, ev_in)
            for l, fn, grid, pack in step["launch"]:
                rtm.launch(fn, grid, l.block, l.smem, pack.array, None)
            self.launch_count += len(step["launch"])
            rtm.event_record(ev_done)
            rtm.stream_wait_event(s_out, ev_done)
            for (name, b, e) in step["d2h"]:
                f = fields[name]
                plane = int(np.prod(f.shape[1:])) if len(f.shape) > 1 else 1
                rtm.d2h(flat[name][(b - base) * plane:(e - base) * plane],
                        self.buffers[name].dptr + (b - base) * plane * f.data_type.bytes, stream=s_out)
                copied[1] += (e - b) * plane * f.data_type.bytes
        rtm.stream_synchronize(s_out)
        rtm.stream_synchronize()
        rtm.event_destroy(start)
        self.last_call_bytes = tuple(copied)           # (host->device, device->host) of this call
        return True

    def __call__(self, **kwargs):
        """Run once with host arrays: copy inputs in, execute, copy outputs back in place.  Large
        programs are cut into pieces along the outermost dimension so that the copies of one piece
        overlap the passes and the copies of its neighbours (``SFB200_PIPELINE_PIECES``, 0 = off)."""
        arrays, scalars = self._split_call_args(kwargs)
        fields = self.program.fields
        pieces = int(os.environ.get("SFB200_PIPELINE_PIECES", "16"))
        in_out = [n for n, f in fields.items() if not f.is_scalar and f.kind in ("input", "output")]
        if (pieces > 1 and self.synthetic_reads is None and all(n in arrays for n in in_out)
                and sum(fields[n].nbytes for n in in_out) >= self.PIPELINE_MIN_BYTES):
            need = [n for n, f in fields.items() if f.is_scalar]
            missing = [n for n in need if n not in scalars and n not in self.scalar_values]
            if missing:
                raise KeyError("scalar input(s) {} were not provided".format(missing))
            if scalars:
                self.set_scalars(scalars)
            if self._call_pipelined(arrays, pieces):
                return
        for name, f in fields.items():
            if f.kind == "input" and not f.is_scalar:
                if self.synthetic_reads is not None:
                    self.rt.fill_constant(self.buffers[name].dptr, int(np.prod(self.local_shape(name))),
                                          f.data_type, self.synthetic_reads)
                elif name in arrays:
                    self.upload(name, arrays[name])
                else:
                    raise KeyError("input array {} was not provided".format(name))
        need = [n for n, f in fields.items() if f.is_scalar]
        missing = [n for n in need if n not in scalars and n not in self.scalar_values]
        if missing:
            raise KeyError("scalar input(s) {} were not provided".format(missing))
        if scalars:
            self.set_scalars(scalars)
        self.execute()
        for name in self.program.outputs:
            if name in arrays:
                self.download(name, arrays[name])
        self.rt.stream_synchronize()

    def time_execution(self, repetitions=10, warmup=3, graph=False):
        """Device time (ms, list) of ``repetitions`` executions, CUDA events on the launch stream."""
        run = self.execute_graph if graph else self.execute
        for _ in range(warmup):
            run()
        self.rt.stream_synchronize()
        times = []
        e0, e1 = self.rt.event_create(), self.rt.event_create()
        for _ in range(repetitions):
            self.rt.event_record(e0)
            run()
            self.rt.event_record(e1)
            self.rt.event_synchronize(e1)
            times.append(self.rt.elapsed_ms(e0, e1))
        self.rt.event_destroy(e0)
        self.rt.event_destroy(e1)
        return times
