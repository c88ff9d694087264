"""Host side of the decode op: torch tensors in, packed detection tensors out.

``sdnet_b200::decode`` is a ``torch.library`` custom op whose implementation is one
ctypes call into the ``extern "C"`` launcher ``sdnet_decode_launch`` on torch's current
CUDA stream.  torch is used for device memory, streams and op registration only; all
arithmetic happens in the hand-written sm_100a kernels.  There is no CPU or eager
fallback: CPU tensors are rejected and a missing library raises at first use.

Replaces (reference): src/sdnet/data/decoders.py:44-100 and the helpers it calls in
src/sdnet/utils/utils.py:342-361,422-467.
"""
from __future__ import annotations

import ctypes
import math
from collections.abc import Mapping
from dataclasses import dataclass

import torch

from . import _native
PEAKS_PATHS = ("warp", "tile", "tile_row_pairs")  # SDNET_PATH_* in include/sdnet_decode.h
from ._native import (FLAG_EXACT_SELECT, FLAG_NO_GROUPING, FLAG_PRE_ACTIVATED, FLAG_WARP_KERNEL, FLAG_WORKSPACE_CLEAN,
                      SdnetDecodeParams,
                      SdnetSchedule, SdnetTensor4)

__all__ = ["decode_packed", "activate_maps", "suppress_maps", "suppress_into", "DecodePlan", "DecodePipeline",
           "PackedDetections", "gpu_launches_per_decode", "class_thresholds"]

# kernels launched by one sdnet_decode_launch: peaks, exact-select, tail (+ one memset node)
_KERNELS_PER_DECODE = 3


def gpu_launches_per_decode() -> int:
    return _KERNELS_PER_DECODE


def _view4(t: torch.Tensor) -> SdnetTensor4:
    sb, sc, sh, sw = t.stride()
    return SdnetTensor4(t.data_ptr(), sb, sc, sh, sw)


_DTYPES = {torch.float32: _native.DTYPE_F32, torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}


def _check_tensor(name: str, t: torch.Tensor, allow_pinned_host: bool = False, dtype: torch.dtype | None = None):
    """Device / rank / dtype checks.  fp32, fp16 and bf16 are accepted: the reference computes the
    sigmoid in the input dtype, and so do the kernels; nothing is ever upcast silently."""
    if t.dtype not in _DTYPES:
        raise TypeError(f"{name}: dtype {t.dtype} is not supported by the B200 decode path (float32, float16, bfloat16)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name}: dtype {t.dtype} differs from anchor_hm's {dtype}; the four network outputs are views "
                        "of one tensor in the reference and must share a dtype")
    if t.dim() != 4:
        raise ValueError(f"{name}: expected a (B, C, H, W) tensor, got shape {tuple(t.shape)}")
    if not t.is_cuda and not (allow_pinned_host and t.is_pinned()):
        raise RuntimeError(
            f"{name} lives on {t.device}: the B200 decode path has no CPU fallback "
            "(move the network outputs to a CUDA device)"
        )


@dataclass
class PackedDetections:
    """Device tensors produced by one decode (layouts: include/sdnet_decode.h)."""

    anchor_out: torch.Tensor  # (B, K, 4) x, y, score, class
    part_out: torch.Tensor  # (B, P, 6) x, y, score, kind, origin_x, origin_y
    anchor_inds: torch.Tensor  # (B, K) int64
    part_inds: torch.Tensor  # (B, P) int64
    part_emb: torch.Tensor  # (B, P, 2)
    assign: torch.Tensor  # (B, P) int32, -1 = not grouped
    counts: torch.Tensor  # (B, 2) int32
    diag: torch.Tensor  # (B*(M+N), 2) int32
    blob: torch.Tensor | None = None  # the single allocation the fields above are views of

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k in
                ("anchor_out", "part_out", "anchor_inds", "part_inds", "part_emb", "assign", "counts", "diag")}


def _carve(blob: torch.Tensor, B: int, K: int, P: int, C: int) -> PackedDetections:
    """Views of one uint8 allocation, 8-byte fields first so every view is aligned."""
    off = 0

    def take(nbytes, dtype, shape):
        nonlocal off
        view = blob[off : off + nbytes].view(dtype).view(shape)
        off += (nbytes + 15) // 16 * 16
        return view

    a_inds = take(B * K * 8, torch.int64, (B, K))
    p_inds = take(B * P * 8, torch.int64, (B, P))
    a_out = take(B * K * 16, torch.float32, (B, K, 4))
    p_out = take(B * P * 24, torch.float32, (B, P, 6))
    p_emb = take(B * P * 8, torch.float32, (B, P, 2))
    assign = take(B * P * 4, torch.int32, (B, P))
    counts = take(B * 8, torch.int32, (B, 2))
    diag = take(B * C * 8, torch.int32, (B * C, 2))
    return PackedDetections(a_out, p_out, a_inds, p_inds, p_emb, assign, counts, diag, blob)


def packed_nbytes(B: int, K: int, P: int, C: int) -> int:
    sizes = (B * K * 8, B * P * 8, B * K * 16, B * P * 24, B * P * 8, B * P * 4, B * 8, B * C * 8)
    return sum((s + 15) // 16 * 16 for s in sizes)


class DecodePlan:
    """Pre-sized workspace + output blob for one (device, shape, K, P): the low-overhead way
    to call the C ABI repeatedly (bench loop, CUDA-graph capture, sharded decode)."""

    def __init__(self, device, B, M, N, H, W, K, P, dtype: torch.dtype = torch.float32, lib=None):
        self.shape = (B, M, N, H, W, K, P)
        self.dtype = dtype
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.lib = lib if lib is not None else _native.load()
        self.workspace_bytes = _native.workspace_bytes(B, M, N, H, W, K, P, _DTYPES[dtype], lib=self.lib)
        self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
        self.out = _carve(torch.empty(packed_nbytes(B, K, P, M + N), dtype=torch.uint8, device=self.device),
                          B, K, P, M + N)
        self.params = SdnetDecodeParams()
        p = self.params
        p.struct_size = ctypes.sizeof(SdnetDecodeParams)
        p.dtype = _DTYPES[dtype]
        p.B, p.M, p.N, p.H, p.W, p.K, p.P = B, M, N, H, W, K, P
        p.workspace = self.workspace.data_ptr()
        p.workspace_bytes = self.workspace_bytes
        self._bind_outputs(self.out)
        self._clean = False  # True once a decode has run on this workspace: its tail kernel leaves the header zeroed

    def _launch(self, fn, *args) -> None:
        """Call a launch entry point; after the first successful decode the per-call memset of the workspace header is
        skipped (SDNET_FLAG_WORKSPACE_CLEAN: every decode zeroes the header behind itself)."""
        if self._clean:
            self.params.flags |= FLAG_WORKSPACE_CLEAN
        rc = fn(ctypes.byref(self.params), *args)
        self._clean = rc == 0
        _native.check(rc, fn.__name__)

    def _bind_outputs(self, out: PackedDetections):
        p = self.params
        p.anchor_out, p.part_out = out.anchor_out.data_ptr(), out.part_out.data_ptr()
        p.anchor_inds, p.part_inds = out.anchor_inds.data_ptr(), out.part_inds.data_ptr()
        p.part_emb, p.assign = out.part_emb.data_ptr(), out.assign.data_ptr()
        p.counts, p.diag = out.counts.data_ptr(), out.diag.data_ptr()

    def _check_inputs(self, anchor_hm, part_hm, offsets, embeddings, host_ok: bool = False):
        """The kernels trust the plan's (B, M, N, H, W), dtype and device: a tensor that differs would be
        reinterpreted or read out of bounds, so refuse it here."""
        B, M, N, H, W, _, _ = self.shape
        want = (("anchor_hm", anchor_hm, M), ("part_hm", part_hm, N), ("offsets", offsets, 2), ("embeddings", embeddings, 2))
        for name, t, channels in want:
            if t is None:
                continue
            if t.dtype != self.dtype:
                raise TypeError(f"{name}: dtype {t.dtype} differs from the plan's {self.dtype}")
            if tuple(t.shape) != (B, channels, H, W):
                raise ValueError(f"{name}: shape {tuple(t.shape)} differs from the plan's {(B, channels, H, W)}")
            if t.is_cuda:
                if t.device != self.device:
                    raise RuntimeError(f"{name} lives on {t.device}, the plan on {self.device}")
            elif not (host_ok and t.is_pinned()):
                raise RuntimeError(f"{name} lives on {t.device}: the B200 decode path has no CPU fallback")

    def _check_conf_class(self, conf_class):
        """The tail kernel reads M + N fp32 thresholds from the table's device pointer: refuse anything else."""
        _, M, N = self.shape[:3]
        if conf_class.dtype != torch.float32 or conf_class.dim() != 1 or conf_class.numel() != M + N:
            raise ValueError(f"conf_class: expected a 1-D float32 tensor of M + N = {M + N} thresholds, got "
                             f"{conf_class.dtype} of shape {tuple(conf_class.shape)}")
        if not conf_class.is_cuda or conf_class.device != self.device or not conf_class.is_contiguous():
            raise ValueError(f"conf_class must be a contiguous tensor on {self.device}, not on {conf_class.device}")

    def _bind_inputs(self, anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags,
                     host_ok: bool = False, conf_class=None):
        self._check_inputs(anchor_hm, part_hm, offsets, embeddings, host_ok)
        if conf_class is not None:
            self._check_conf_class(conf_class)
        p = self.params
        p.anchor_hm, p.part_hm, p.offsets = _view4(anchor_hm), _view4(part_hm), _view4(offsets)
        p.embeddings = _view4(embeddings) if embeddings is not None else SdnetTensor4(None, 0, 0, 0, 1)
        p.conf_f32, p.dist_abs_f32 = conf_f32, dist_abs_f32
        p.conf_class_f32 = conf_class.data_ptr() if conf_class is not None else None
        p.radius, p.flags = radius, flags

    def run(self, anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius=2, flags=0,
            stream=None, conf_class=None) -> PackedDetections:
        """Enqueue one decode on ``stream`` (a torch stream or raw handle; default: torch's current stream). Asynchronous.
        ``conf_class``: optional per-class thresholds, a float32 tensor of M + N entries on the plan's device (anchor
        classes, then part kinds; each rounded to the heat maps' dtype) used instead of ``conf_f32``."""
        self._bind_inputs(anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags,
                          conf_class=conf_class)
        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        stream = getattr(stream, "cuda_stream", stream)  # a torch.cuda.Stream or a raw cudaStream_t
        self._launch(self.lib.sdnet_decode_launch, ctypes.c_void_p(stream))
        return self.out

    def peaks_path(self, anchor_hm, part_hm, offsets, embeddings, radius=2, flags=0) -> str:
        """Which peaks kernel these tensors would run: "warp" | "tile" | "tile_row_pairs"."""
        self._bind_inputs(anchor_hm, part_hm, offsets, embeddings, 0.0, 0.0, radius, flags)
        rc = self.lib.sdnet_decode_peaks_path(ctypes.byref(self.params))
        if rc < 0:  # non-negative values are SDNET_PATH_*, not CUDA errors
            _native.check(rc, "sdnet_decode_peaks_path")
        return PEAKS_PATHS[rc]

    def schedule(self, anchor_hm, part_hm, offsets, embeddings, radius=2, flags=0) -> dict:
        """How the peaks kernel cuts these tensors into units on this device (``sdnet_decode_schedule``)."""
        self._bind_inputs(anchor_hm, part_hm, offsets, embeddings, 0.0, 0.0, radius, flags)
        out = SdnetSchedule()
        out.struct_size = ctypes.sizeof(SdnetSchedule)
        with torch.cuda.device(self.device):
            rc = self.lib.sdnet_decode_schedule(ctypes.byref(self.params), ctypes.byref(out))
        _native.check(rc, "sdnet_decode_schedule")
        d = {name: getattr(out, name) for name, _ in SdnetSchedule._fields_ if name != "struct_size"}
        d["path"] = PEAKS_PATHS[d["path"]]
        return d

    def run_timed(self, anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius=2, flags=0,
                  conf_class=None):
        """Synchronous profiling run: returns (peaks_ms, exact_select_ms, tail_ms) device times."""
        self._bind_inputs(anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags,
                          conf_class=conf_class)
        ms = (ctypes.c_float * 3)()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._launch(self.lib.sdnet_decode_launch_timed, ctypes.c_void_p(stream), ms)
        return tuple(float(x) for x in ms)

    def run_host(self, anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, staging: torch.Tensor,
                 radius=2, flags=0, stream=None, conf_class=None) -> PackedDetections:
        """Same, with the four inputs in pinned HOST memory (``sdnet_decode_host_launch``); ``conf_class`` stays a
        device tensor."""
        self._bind_inputs(anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags, host_ok=True,
                          conf_class=conf_class)
        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        stream = getattr(stream, "cuda_stream", stream)
        self._launch(self.lib.sdnet_decode_host_launch, ctypes.c_void_p(staging.data_ptr()),
                     ctypes.c_size_t(staging.numel() * staging.element_size()), ctypes.c_void_p(stream))
        return self.out


class DecodePipeline:
    """Several decodes in flight: ``depth`` plans (each with its own workspace and outputs) on ``depth``
    CUDA streams, used round-robin.  While one batch is in its short, latency-bound tail kernel the next
    batch's peaks kernel already streams its heat maps, so a stream of batches runs at the peaks kernel's
    rate.  ``submit`` returns the slot's outputs and an event; a slot's outputs are overwritten
    ``depth`` submits later, so consume them (or wait on the event and copy) before that.

    Stream safety: ``submit`` makes the slot's stream wait for everything already enqueued on the
    caller's current stream (the producer of the inputs) and tells the caching allocator that the
    inputs are in use on the slot's stream (``record_stream``), so the network may run ahead and
    free/reuse its output buffers without the decode reading recycled memory.

    ``make_plan(i)`` builds slot i's plan: anything with ``.run(..., stream=)`` (``DecodePlan``,
    ``parallel.FusedGatherPlan``)."""

    def __init__(self, device, depth: int, make_plan):
        self.device = torch.device(device)
        self.plans = [make_plan(i) for i in range(depth)]
        self.streams = [torch.cuda.Stream(self.device) for _ in range(depth)]
        self.events = [torch.cuda.Event() for _ in range(depth)]
        self._next = 0

    @classmethod
    def for_shape(cls, device, depth, B, M, N, H, W, K, P, dtype: torch.dtype = torch.float32):
        return cls(device, depth, lambda _i: DecodePlan(device, B, M, N, H, W, K, P, dtype))

    def after(self, event: torch.cuda.Event):
        """Make every slot's stream wait for ``event`` (e.g. the producer of the inputs)."""
        for st in self.streams:
            st.wait_event(event)

    def submit(self, anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius=2, flags=0,
               conf_class=None):
        """``conf_class``: as ``DecodePlan.run``; only plans that take it (``DecodePlan``) accept a table."""
        k = self._next
        self._next = (k + 1) % len(self.plans)
        self.streams[k].wait_stream(torch.cuda.current_stream(self.device))
        for t in (anchor_hm, part_hm, offsets, embeddings, conf_class):
            if t is not None and t.is_cuda:
                t.record_stream(self.streams[k])
        extra = {} if conf_class is None else {"conf_class": conf_class}
        out = self.plans[k].run(anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags,
                                stream=self.streams[k], **extra)
        self.events[k].record(self.streams[k])
        return out, self.events[k]

    def drain(self, stream: torch.cuda.Stream | None = None):
        """Make ``stream`` (default: the current one) wait for everything submitted so far."""
        stream = stream if stream is not None else torch.cuda.current_stream(self.device)
        for plan, st in zip(self.plans, self.streams):
            arrived = getattr(plan, "wait_arrival", None)  # parallel.FusedGatherPlan in lazy mode: the gather's arrival
            if arrived is not None:
                arrived(st)
            stream.wait_stream(st)


def _f32(value: float, dtype: torch.dtype = torch.float32) -> float:
    """Round a Python double to `dtype` the way torch does when a tensor of that dtype is compared
    with a scalar (the result is exactly representable in fp32 for every supported dtype)."""
    return float(torch.tensor(value, dtype=dtype))


def class_thresholds(conf_thresh, class_names, kind_names, default) -> float | list[float]:
    """A decoder or evaluator threshold as the kernels take it: a number stays a number; a mapping from class or part
    kind name to threshold becomes one threshold per anchor class, then one per part kind.  ``class_names`` /
    ``kind_names``: the name of each class / kind index (``None`` for an index without a name); a name the mapping
    leaves out takes ``default``.  A name that is both a class and a kind sets both.  Raises ``ValueError`` for a name
    that is neither and for a threshold that is not finite."""
    if not isinstance(conf_thresh, Mapping):
        return float(conf_thresh)
    known = set(class_names) | set(kind_names)
    unknown = [name for name in conf_thresh if name is None or name not in known]
    if unknown:
        raise ValueError(f"conf_thresh names {unknown!r}, which are neither classes {[n for n in class_names if n is not None]} "
                         f"nor part kinds {[n for n in kind_names if n is not None]}")
    table = {name: float(value) for name, value in conf_thresh.items()}
    bad = {name: value for name, value in table.items() if not math.isfinite(value)}
    if bad:
        raise ValueError(f"conf_thresh values must be finite: {bad!r}")
    default = float(default)
    return [table.get(name, default) if name is not None else default for name in (*class_names, *kind_names)]


def _conf_arg(conf_thresh, M: int, N: int, dtype: torch.dtype, device) -> tuple[float, torch.Tensor | None]:
    """(conf_f32, conf_class) of a decode: one threshold, or M + N per-class thresholds (anchor classes, then part
    kinds) as a device table, each rounded to the heat maps' dtype like the scalar."""
    if not isinstance(conf_thresh, (list, tuple)) and getattr(conf_thresh, "ndim", 0) == 0:
        return _f32(float(conf_thresh), dtype), None
    values = [float(v) for v in (conf_thresh.tolist() if hasattr(conf_thresh, "tolist") else conf_thresh)]
    if len(values) != M + N:
        raise ValueError(f"per-class conf_thresh has {len(values)} entries; the heat maps have M + N = {M + N} classes")
    if not all(math.isfinite(v) for v in values):
        raise ValueError("per-class conf_thresh values must be finite")
    return 0.0, torch.tensor([_f32(v, dtype) for v in values], dtype=torch.float32).to(device)


# ------------------------------------------------------------------------------------ custom ops
_OP_PLANS: dict = {}
_OP_PLANS_MAX = 8


def _op_plan(device, B, M, N, H, W, K, P, dtype) -> DecodePlan:
    """Workspace cache of the custom op, keyed by (device, stream, shape, dtype): a decode needs its
    scratch only while its three kernels run, and work on one stream is ordered, so consecutive calls
    on a stream share one workspace instead of allocating ~0.1 MB per image per call."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, B, M, N, H, W, K, P, dtype)
    plan = _OP_PLANS.get(key)
    if plan is None:
        if len(_OP_PLANS) >= _OP_PLANS_MAX:
            _OP_PLANS.pop(next(iter(_OP_PLANS)))
        plan = _OP_PLANS[key] = DecodePlan(device, B, M, N, H, W, K, P, dtype)
    return plan


@torch.library.custom_op("sdnet_b200::decode", mutates_args=(), device_types="cuda")
def _decode_op(anchor_hm: torch.Tensor, part_hm: torch.Tensor, offsets: torch.Tensor, embeddings: torch.Tensor,
               max_objects: int, max_parts: int, conf_f32: float, dist_abs_f32: float, radius: int,
               flags: int, conf_class: torch.Tensor | None = None) -> torch.Tensor:
    B, M, H, W = anchor_hm.shape
    N = part_hm.shape[1]
    with torch.cuda.device(anchor_hm.device):
        plan = _op_plan(anchor_hm.device, B, M, N, H, W, max_objects, max_parts, anchor_hm.dtype)
        # the op returns a fresh tensor (no aliasing between calls); the workspace is the cached part
        blob = torch.empty(plan.out.blob.numel(), dtype=torch.uint8, device=anchor_hm.device)
        plan._bind_outputs(_carve(blob, B, max_objects, max_parts, M + N))
        plan.run(anchor_hm, part_hm, offsets, embeddings, conf_f32, dist_abs_f32, radius, flags, conf_class=conf_class)
    return blob


@_decode_op.register_fake
def _(anchor_hm, part_hm, offsets, embeddings, max_objects, max_parts, conf_f32, dist_abs_f32, radius, flags,
      conf_class=None):
    B, M = anchor_hm.shape[:2]
    N = part_hm.shape[1]
    return anchor_hm.new_empty(packed_nbytes(B, max_objects, max_parts, M + N), dtype=torch.uint8)


@torch.library.custom_op("sdnet_b200::activate", mutates_args=(), device_types="cuda")
def _activate_op(hm: torch.Tensor) -> torch.Tensor:
    B, C, H, W = hm.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=hm.device)
    view = _view4(hm)
    with torch.cuda.device(hm.device):
        rc = _native.load().sdnet_activate_launch(ctypes.byref(view), _DTYPES[hm.dtype], B, C, H, W,
                                                  ctypes.c_void_p(out.data_ptr()),
                                                  ctypes.c_void_p(torch.cuda.current_stream(hm.device).cuda_stream))
    _native.check(rc, "sdnet_activate_launch")
    return out


@_activate_op.register_fake
def _(hm):
    return hm.new_empty(hm.shape, dtype=torch.float32)


@torch.library.custom_op("sdnet_b200::suppress", mutates_args=(), device_types="cuda")
def _suppress_op(hm: torch.Tensor, radius: int) -> torch.Tensor:
    B, C, H, W = hm.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=hm.device)
    view = _view4(hm)
    with torch.cuda.device(hm.device):
        rc = _native.load().sdnet_suppress_launch(ctypes.byref(view), _DTYPES[hm.dtype], B, C, H, W, radius,
                                                  ctypes.c_void_p(out.data_ptr()),
                                                  ctypes.c_void_p(torch.cuda.current_stream(hm.device).cuda_stream))
    _native.check(rc, "sdnet_suppress_launch")
    return out


@_suppress_op.register_fake
def _(hm, radius):
    return hm.new_empty(hm.shape, dtype=torch.float32)


@torch.library.custom_op("sdnet_b200::suppress_into", mutates_args=("out",), device_types="cuda")
def _suppress_into_op(hm: torch.Tensor, out: torch.Tensor, radius: int) -> None:
    B, C, H, W = hm.shape
    view, oview = _view4(hm), _view4(out)
    with torch.cuda.device(hm.device):
        rc = _native.load().sdnet_suppress_into_launch(ctypes.byref(view), _DTYPES[hm.dtype], B, C, H, W, radius, ctypes.byref(oview),
                                                       ctypes.c_void_p(torch.cuda.current_stream(hm.device).cuda_stream))
    _native.check(rc, "sdnet_suppress_into_launch")


def _unit_w_stride(t: torch.Tensor) -> torch.Tensor:
    # a layout fix on the device, not a fallback: the kernels need the innermost stride to be 1
    return t if t.stride(3) == 1 else t.contiguous()


def decode_packed(outputs: dict, max_objects: int, max_parts: int, conf_thresh, dist_thresh: float, *,
                  pre_activated: bool = False, group: bool = True, radius: int = 2,
                  exact_select: bool = False, warp_kernel: bool = False) -> PackedDetections:
    """Run the CUDA decode on the four network-output views and return packed device tensors.

    ``conf_thresh``: one threshold, or a sequence of M + N per-class thresholds -- one per anchor class (heat-map
    channel), then one per part kind -- each slot compared against the entry of its own class (``class_thresholds``
    builds one from a name mapping).  Only ``counts`` and the grouping depend on it."""
    a_hm, p_hm, off = outputs["anchor_hm"], outputs["part_hm"], outputs["offsets"]
    emb = outputs["embeddings"] if group or "embeddings" in outputs else None
    on_host = not a_hm.is_cuda  # pinned host tensors take the host-buffer entry point (everything else on a CPU raises)
    for name, t in (("anchor_hm", a_hm), ("part_hm", p_hm), ("offsets", off)) + ((("embeddings", emb),) if emb is not None else ()):
        _check_tensor(name, t, allow_pinned_host=on_host, dtype=a_hm.dtype)
        if t.is_cuda == on_host:
            raise RuntimeError(f"{name} lives on {t.device} but anchor_hm on {a_hm.device}: keep the four outputs together")
    B, M, H, W = a_hm.shape
    N = p_hm.shape[1]
    if emb is None:
        emb = off  # never read under NO_GROUPING without part_emb consumers; keeps the op signature tensor-only
    flags = (FLAG_PRE_ACTIVATED if pre_activated else 0) | (0 if group else FLAG_NO_GROUPING) | (
        FLAG_EXACT_SELECT if exact_select else 0) | (FLAG_WARP_KERNEL if warp_kernel else 0)
    # `scores > conf` compares in the scores' dtype (fp16 scores against fp16(conf)); the distance gate
    # always compares fp32 distances
    device = a_hm.device if not on_host else torch.device("cuda", torch.cuda.current_device())
    conf_f32, conf_class = _conf_arg(conf_thresh, M, N, a_hm.dtype, device)
    if on_host:
        return _decode_from_host(a_hm, p_hm, off, emb, int(max_objects), int(max_parts),
                                 conf_f32, _f32(float(dist_thresh) * min(W, H)), int(radius), int(flags), conf_class)
    a_hm, p_hm, off, emb = map(_unit_w_stride, (a_hm, p_hm, off, emb))
    blob = _decode_op(a_hm, p_hm, off, emb, int(max_objects), int(max_parts), conf_f32,
                      _f32(float(dist_thresh) * min(W, H)), int(radius), int(flags), conf_class)
    return _carve(blob, B, int(max_objects), int(max_parts), M + N)


def _decode_from_host(a_hm, p_hm, off, emb, K, P, conf_f32, dist_abs_f32, radius, flags, conf_class=None) -> PackedDetections:
    """Pinned HOST tensors -> packed detections on the current CUDA device (``sdnet_decode_host_launch``:
    the heat planes are uploaded into a cached staging buffer, offsets/embeddings are read in place)."""
    B, M, H, W = a_hm.shape
    N = p_hm.shape[1]
    device = torch.device("cuda", torch.cuda.current_device())
    plan = _op_plan(device, B, M, N, H, W, K, P, a_hm.dtype)
    need = B * (M + N) * H * W * a_hm.element_size()
    if getattr(plan, "staging", None) is None or plan.staging.numel() < need:
        plan.staging = torch.empty(need, dtype=torch.uint8, device=device)
    blob = torch.empty(plan.out.blob.numel(), dtype=torch.uint8, device=device)
    out = _carve(blob, B, K, P, M + N)
    plan._bind_outputs(out)
    plan.run_host(a_hm, p_hm, off, emb, conf_f32, dist_abs_f32, plan.staging, radius, flags, conf_class=conf_class)
    return out


def peaks_path(outputs: dict, max_objects: int, max_parts: int, *, radius: int = 2, warp_kernel: bool = False) -> str:
    """Name of the peaks kernel ``decode_packed`` runs for these tensors (host-only query)."""
    a_hm, p_hm, off, emb = map(_unit_w_stride, (outputs["anchor_hm"], outputs["part_hm"], outputs["offsets"],
                                                outputs["embeddings"]))
    B, M, H, W = a_hm.shape
    plan = DecodePlan(a_hm.device, B, M, p_hm.shape[1], H, W, int(max_objects), int(max_parts), a_hm.dtype)
    return plan.peaks_path(a_hm, p_hm, off, emb, radius, FLAG_WARP_KERNEL if warp_kernel else 0)


def activate_maps(hm: torch.Tensor) -> torch.Tensor:
    """``clamp(sigmoid(hm), 1e-6, 1-1e-6)`` as a contiguous tensor of hm's dtype (reference utils.py:355-361)."""
    _check_tensor("heat map", hm)
    out = _activate_op(_unit_w_stride(hm))  # fp32 storage of values exactly representable in hm.dtype
    return out if hm.dtype == torch.float32 else out.to(hm.dtype)


def suppress_into(hm: torch.Tensor, out: torch.Tensor, radius: int = 2) -> torch.Tensor:
    """``nms(clamped_sigmoid(hm))`` written into ``out``, a float32 ``(B, C, H, W)`` view with unit innermost stride
    (e.g. the first channels of a wider tensor): no intermediate tensor, no ``torch.cat`` afterwards."""
    _check_tensor("heat map", hm)
    if out.dtype != torch.float32 or out.shape != hm.shape or out.device != hm.device or out.stride(3) != 1:
        raise ValueError("out must be a float32 view of hm's shape on hm's device with unit innermost stride")
    _suppress_into_op(_unit_w_stride(hm), out, int(radius))
    return out


def suppress_maps(hm: torch.Tensor, radius: int = 2) -> torch.Tensor:
    """``nms(clamped_sigmoid(hm))`` (reference utils.py:355-361,441-443) as a contiguous tensor of hm's dtype:
    the score at the peaks of every (2 radius + 1)^2 window, 0 elsewhere."""
    _check_tensor("heat map", hm)
    out = _suppress_op(_unit_w_stride(hm), int(radius))
    return out if hm.dtype == torch.float32 else out.to(hm.dtype)
