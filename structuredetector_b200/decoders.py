"""Drop-in decoders: same constructor, call signature and return structure as the reference
(reference: src/sdnet/data/decoders.py:17-179 ``Decoder``, 182-342 ``CoreMLDecoder``,
345-423 ``KeypointDecoder``), with the tensor half running in the sm_100a kernels.

What stays in Python is what the reference also does on the host: turning K+P packed
rows per image into ``ImageAnnotation`` objects.  The reference reads every scalar with
``.item()`` (~1,000 device syncs per image); here the packed result comes back in ONE
device->host copy and the objects are built from ``.tolist()`` rows.
"""
from __future__ import annotations

import contextlib
import gc
import json
from pathlib import Path

import numpy as np
import torch

from . import ops
from .annotations import ImageAnnotation, Keypoint, Object

try:
    from . import _fastobj  # C object assembly (csrc/fastobj.c), built by structuredetector_b200.build
except ImportError as exc:  # no silent slow path: say how to get it
    raise ImportError("structuredetector_b200._fastobj is missing: run `python structuredetector_b200/build.py` "
                      "(gcc, CPython headers) to build the object-assembly extension") from exc

__all__ = ["Decoder", "CoreMLDecoder", "KeypointDecoder", "RawDecoder", "CoreMLModel"]


@contextlib.contextmanager
def _gc_paused():
    """Building ~300 small acyclic objects per image makes the cyclic collector re-scan an ever larger
    young generation (measured: 1.3 k -> 4.0 k images/s on dense outputs with it paused)."""
    was_enabled = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was_enabled:
            gc.enable()


class _DecoderBase:
    _pre_activated = False

    def __init__(self, args):
        # the eight fields the reference decoder reads (decoders.py:19-26, 33-38)
        self.label_map = args._r_labels
        self.part_map = args._r_parts
        self.anchor_name = args.anchor_name
        self.args = args
        self.down_ratio = args.down_ratio
        self.max_objects = args.max_objects  # K
        self.max_parts = args.max_parts  # P

    # -- helpers ---------------------------------------------------------------------------
    def _sizes(self, outputs):
        out_h, out_w = outputs["anchor_hm"].shape[2:]
        in_h, in_w = int(self.down_ratio * out_h), int(self.down_ratio * out_w)
        return (out_w, out_h), (in_w, in_h)

    @staticmethod
    def _to_host(packed: ops.PackedDetections) -> ops.PackedDetections:
        """One device->host copy of the whole packed result."""
        blob = packed.blob.cpu()
        b, k = packed.anchor_inds.shape
        p = packed.part_inds.shape[1]
        return ops._carve(blob, b, k, p, packed.diag.shape[0] // b)


class Decoder(_DecoderBase):
    """``decoder(outputs, conf_thresh=None, dist_thresh=None, return_metadata=False)``.

    ``conf_thresh`` may also be a mapping from class or part kind name (``args._r_labels`` / ``args._r_parts``) to
    threshold, e.g. ``ThresholdSweep.best_thresholds()``: every compare against the threshold then uses the entry of
    the slot's own class, and a name the mapping leaves out takes ``args.conf_threshold``."""

    def _conf(self, outputs, conf_thresh):
        """The threshold as the decode takes it: a number, or M + N per-class thresholds."""
        if conf_thresh is None:
            return float(self.args.conf_threshold)
        M, N = outputs["anchor_hm"].shape[1], outputs["part_hm"].shape[1]
        names = lambda mapping, n: [mapping.get(i) for i in range(n)]
        return ops.class_thresholds(conf_thresh, names(self.label_map, M), names(self.part_map, N), self.args.conf_threshold)

    def __call__(self, outputs, conf_thresh=None, dist_thresh=None, return_metadata=False):
        conf_thresh = self._conf(outputs, conf_thresh)
        dist_thresh = self.args.decoder_dist_thresh if dist_thresh is None else dist_thresh
        out_size, in_size = self._sizes(outputs)

        packed = ops.decode_packed(outputs, self.max_objects, self.max_parts, conf_thresh, dist_thresh,
                                   pre_activated=self._pre_activated)
        host = self._to_host(packed)
        host_conf = self._host_conf(conf_thresh, outputs["anchor_hm"].shape[1])
        with _gc_paused():
            annotations = self._assemble(host, host_conf, out_size, in_size)
        if not return_metadata:
            return annotations

        meta = {"annotation": annotations}
        if not self._pre_activated:
            meta["anchor_hm_sig"] = ops.activate_maps(outputs["anchor_hm"])
            meta["part_hm_sig"] = ops.activate_maps(outputs["part_hm"])
        a, p = packed.anchor_out, packed.part_out
        # the reference re-binds the score tensors to their masked (-1) versions before
        # returning them (decoders.py:79,84 then 166-173): kept, oddity included
        in_dtype = outputs["anchor_hm"].dtype
        conf32 = torch.tensor(conf_thresh, dtype=in_dtype, device=a.device).float()  # compared in the scores' dtype
        a_conf = p_conf = conf32
        if conf32.dim() == 1:  # each slot against its own class's threshold: anchor classes first, then part kinds
            a_conf, p_conf = conf32[a[..., 3].long()], conf32[outputs["anchor_hm"].shape[1] + p[..., 3].long()]
        mask = lambda s, conf: torch.where(s > conf, s, torch.full_like(s, -1.0))
        meta["embeddings"] = packed.part_emb if in_dtype == torch.float32 else packed.part_emb.to(in_dtype)
        meta["topk_anchor"] = (mask(a[..., 2], a_conf), packed.anchor_inds, a[..., 3], a[..., 1], a[..., 0])
        meta["topk_kp"] = (mask(p[..., 2], p_conf), packed.part_inds, p[..., 3], p[..., 1], p[..., 0])
        with _gc_paused():
            meta["raw_parts"] = self._raw_parts(host, host_conf, out_size, in_size)
        meta["raw_embeddings"] = outputs["embeddings"]
        meta["raw_offsets"] = outputs["offsets"]
        return meta

    # reference: utils.py:275-286 (json_repr / save_json) on what decoders.py:103-139 would have built
    def detections_json(self, outputs, conf_thresh=None, dist_thresh=None, *, image_paths=None, img_sizes=None, net_size=None):
        """One JSON document per image, byte-identical to ``json.dumps(annotation.json_repr(), indent=2)`` of the
        annotations ``self(outputs)`` returns -- written straight from the packed detections by the C loop in
        ``csrc/fastobj.c``, no ``ImageAnnotation`` / ``Object`` / ``Keypoint`` is built.

        With ``img_sizes`` (one ``(w, h)`` per image) and ``net_size = (args.width, args.height)`` the documents are
        those of the reference's ``detect`` loop (cli/detect.py:41-52): the annotation resized from the network input
        to the original image, ``img_size`` and ``image_path`` set.  ``image_paths`` default to ``batch_<i>``.
        ``conf_thresh``: as for ``__call__``, a number or a name mapping."""
        conf_thresh = self._conf(outputs, conf_thresh)
        dist_thresh = self.args.decoder_dist_thresh if dist_thresh is None else dist_thresh
        out_size, in_size = self._sizes(outputs)
        packed = ops.decode_packed(outputs, self.max_objects, self.max_parts, conf_thresh, dist_thresh,
                                   pre_activated=self._pre_activated)
        return self._json_from_host(self._to_host(packed), self._host_conf(conf_thresh, outputs["anchor_hm"].shape[1]), out_size,
                                    in_size, image_paths, img_sizes, net_size)

    def _json_from_host(self, host, conf_thresh, out_size, in_size, image_paths=None, img_sizes=None, net_size=None):
        B, K = host.anchor_out.shape[:2]
        paths = [Path(f"batch_{b}") for b in range(B)] if image_paths is None else [Path(p) for p in image_paths]
        sizes = [None] * B if img_sizes is None else list(img_sizes)
        if len(paths) != B or len(sizes) != B:
            raise ValueError(f"{B} images but {len(paths)} paths / {len(sizes)} image sizes")
        if any(size is not None for size in sizes) and net_size is None:
            raise ValueError("img_sizes need net_size = (args.width, args.height), the frame the decoder's coordinates are in")
        # Keypoint.resize(in_size=net_size, out_size=img_size): x *= img_w / net_w (utils.py:19-26)
        resize = [None if size is None else (size[0] / net_size[0], size[1] / net_size[1]) for size in sizes]
        enc = lambda names: [None if name is None else json.dumps(name) for name in names]
        return _fastobj.json_text(
            host.anchor_out.contiguous().numpy(), host.part_out.contiguous().numpy(), host.assign.contiguous().numpy(), B, K,
            host.part_out.shape[1], self._side(conf_thresh, 0), in_size[0] / out_size[0], in_size[1] / out_size[1], resize,
            enc(self._names(self.label_map)), enc(self._names(self.part_map)), json.dumps(self.anchor_name),
            [json.dumps(str(path.expanduser().resolve())) for path in paths],
            [json.dumps(None if size is None else list(size), indent=2).replace("\n", "\n  ") for size in sizes])

    def save_detections_json(self, outputs, save_dir=None, **kwargs):
        """``detections_json`` written like ``ImageAnnotation.save_json`` (utils.py:282-286): ``<save_dir>/<image stem>.json``."""
        target = Path(save_dir or "detections/")
        target.mkdir(parents=True, exist_ok=True)
        paths = kwargs.get("image_paths")
        texts = self.detections_json(outputs, **kwargs)
        for b, text in enumerate(texts):
            name = Path(paths[b] if paths is not None else f"batch_{b}").with_suffix(".json").name
            (target / name).write_text(text)
        return texts

    # reference: decoders.py:103-139
    def _assemble(self, host: ops.PackedDetections, conf_thresh, out_size, in_size):
        """Python objects from the packed rows, built by the C loop in ``csrc/fastobj.c``: float32 coordinates
        widened to double and multiplied by ``in/out`` in double (the reference multiplies ``.item()`` doubles),
        ``score > conf`` in double, parts bucketed by anchor slot in part-slot order.  ``conf_thresh``: a number, or
        (thresholds of the anchor classes, thresholds of the part kinds)."""
        sx, sy = in_size[0] / out_size[0], in_size[1] / out_size[1]
        a, p, assign = host.anchor_out, host.part_out, host.assign
        B, K = a.shape[:2]
        return _fastobj.assemble(a.contiguous().numpy(), p.contiguous().numpy(), assign.contiguous().numpy(), B, K,
                                 p.shape[1], self._side(conf_thresh, 0), sx, sy, self._names(self.label_map),
                                 self._names(self.part_map), self.anchor_name, Keypoint, Object, ImageAnnotation)

    @staticmethod
    def _host_conf(conf_thresh, M):
        """What the host loops compare scores with: the number, or (anchor classes' thresholds, part kinds')."""
        return (conf_thresh[:M], conf_thresh[M:]) if isinstance(conf_thresh, list) else float(conf_thresh)

    @staticmethod
    def _side(conf_thresh, side):
        """The anchors' (side 0) or the parts' (side 1) threshold argument of the host loops."""
        return conf_thresh[side] if isinstance(conf_thresh, tuple) else float(conf_thresh)

    @staticmethod
    def _names(mapping):
        """Class index -> name as a list (dict lookups with int keys, hoisted out of the loops)."""
        if not mapping:
            return []
        table = [None] * (max(mapping) + 1)
        for index, name in mapping.items():
            table[index] = name
        return table

    # reference: decoders.py:142-159
    def _raw_parts(self, host: ops.PackedDetections, conf_thresh, out_size, in_size):
        sx, sy = in_size[0] / out_size[0], in_size[1] / out_size[1]
        p = host.part_out
        return _fastobj.keypoints(p.contiguous().numpy(), p.shape[0], p.shape[1], p.shape[2], self._side(conf_thresh, 1), sx, sy,
                                  self._names(self.part_map), Keypoint)


class CoreMLDecoder(Decoder):
    """Variant whose heat maps already went through sigmoid + NMS inside the exported model
    (reference: decoders.py:182-342).  Same outputs minus the two ``*_hm_sig`` maps."""

    _pre_activated = True


class KeypointDecoder(_DecoderBase):
    """Keypoints only, no grouping (reference: decoders.py:345-423): returns, per image, the
    anchors then the parts whose fp32 score is not below ``args.conf_threshold``."""

    def __call__(self, outputs):
        conf_thresh = self.args.conf_threshold
        (out_w, out_h), (in_w, in_h) = self._sizes(outputs)
        r_h, r_w = np.float32(in_h / out_h), np.float32(in_w / out_w)
        packed = ops.decode_packed(outputs, self.max_objects, self.max_parts, conf_thresh, 0.0, group=False)
        host = self._to_host(packed)
        with _gc_paused():
            return self._keypoints(host, np.float32(conf_thresh), r_w, r_h)

    def _keypoints(self, host, conf32, r_w, r_h):
        annotations = []
        anchors, parts = host.anchor_out.numpy(), host.part_out.numpy()
        for b in range(anchors.shape[0]):
            keypoints = []
            for rows, names in ((anchors[b], self.label_map), (parts[b], self.part_map)):
                keep = ~(rows[:, 2] < conf32)
                xs = (rows[:, 0] * r_w)[keep].tolist()  # fp32 multiply, as on the reference's tensors
                ys = (rows[:, 1] * r_h)[keep].tolist()
                for x, y, score, cls in zip(xs, ys, rows[keep, 2].tolist(), rows[keep, 3].tolist()):
                    keypoints.append(Keypoint(kind=names[int(cls)], x=x, y=y, score=score))
            annotations.append(keypoints)
        return annotations


class RawDecoder:
    """``RawDecoder(nb_hms)(raw)``: the network's raw ``(B, M+N+4, H, W)`` output with its first ``nb_hms``
    channels replaced by ``nms(clamped_sigmoid(.))`` -- what the reference bakes into its exported model
    (reference: src/sdnet/cli/convert_coreml.py:12-19) and ``CoreMLDecoder`` then consumes.

    float32: ONE kernel writes the baked heat maps straight into the first channels of the result
    (``sdnet_suppress_into_launch``) and the four offset / embedding channels are copied behind them -- the reference's
    sigmoid, clamp, max-pool, compare, multiply and ``torch.cat`` passes (12 reads / writes of the heat maps) become one
    read and one write.  fp16 / bf16 go through a float32 intermediate of the heat maps only."""

    def __init__(self, nb_hms: int) -> None:
        self.nb_hms = nb_hms

    def __call__(self, input: torch.Tensor) -> torch.Tensor:
        n = self.nb_hms
        out = torch.empty(input.shape, dtype=input.dtype, device=input.device)
        if input.dtype == torch.float32:
            ops.suppress_into(input[:, :n], out[:, :n])
        else:
            out[:, :n] = ops.suppress_maps(input[:, :n])
        out[:, n:] = input[:, n:]
        return out


class CoreMLModel(torch.nn.Module):
    """``CoreMLModel(model, args)``: the network followed by ``RawDecoder`` as one module -- sigmoid + NMS fused onto the
    head's output (reference: src/sdnet/cli/convert_coreml.py:21-29).  ``model`` is any module returning the raw
    ``(B, M+N+4, H/4, W/4)`` tensor (the reference ``Network`` with ``raw_output=True``); ``forward`` returns that tensor
    with the heat maps baked, i.e. what ``CoreMLDecoder`` decodes."""

    def __init__(self, model: torch.nn.Module, args) -> None:
        super().__init__()
        self.model = model
        self.decoder = RawDecoder(nb_hms=len(args.labels) + len(args.parts))

    def forward(self, image: torch.Tensor) -> torch.Tensor:
        return self.decoder(self.model(image))
