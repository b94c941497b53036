"""CPU: every mirrored callable keeps the reference's signature -- same parameter
names in the same order with the same defaults (extra trailing keyword parameters are allowed), so the
call sites of the reference's solvers / eval script work unchanged (INTEGRATION.md).

With the reference tree mounted the parameter lists are compared with the reference's own. Without it they are
compared with ``tests/golden/mirrored_signatures.json``: this package's parameter lists as recorded when the record was
added (``SP_RECORD_REFERENCE_PINS=missing`` adds labels that have none). Those lists start with the reference's and
extend it only by parameters with defaults, so keeping them (plus new trailing parameters with defaults) keeps the
reference's."""
import inspect
import json
import os

import pytest

from oracle import ref_loader
from conftest import GOLDEN

RECORD = os.path.join(GOLDEN, "mirrored_signatures.json")


def _params(fn):
    return [(p.name, p.default) for p in inspect.signature(fn).parameters.values() if p.name != "self"]


def _same_default(a, b):
    if a is inspect.Parameter.empty or b is inspect.Parameter.empty:
        return a is b
    try:
        import numpy as np
        if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):      # get_affine_transform(shift=array([0, 0]))
            return b is None or (isinstance(b, np.ndarray) and np.array_equal(a, b))
    except Exception:
        pass
    return a == b


def _check(ref_fn, our_fn, label):
    ref_p, our_p = _params(ref_fn), _params(our_fn)
    assert len(our_p) >= len(ref_p), (label, ref_p, our_p)
    for (rn, rd), (on, od) in zip(ref_p, our_p):
        assert rn == on, (label, rn, on)
        assert _same_default(rd, od), (label, rn, rd, od)
    for name, default in our_p[len(ref_p):]:
        assert default is not inspect.Parameter.empty, (label, "extra parameter without default", name)


def _mirrored():
    """(label, our callable, the reference's callable given the loaded reference)."""
    from simple_pose_b200.commons import joint_utils as ju, transforms as tr
    from simple_pose_b200.datasets import naive_data as nd
    from simple_pose_b200.metrics import pose_metrics as pm
    return [
        ("RefineSimpleTransform()", tr.RefineSimpleTransform.__init__, lambda r: r.transforms.RefineSimpleTransform.__init__),
        ("Refine.get_heat_map", tr.RefineSimpleTransform.get_heat_map, lambda r: r.transforms.RefineSimpleTransform.get_heat_map),
        ("BasicSimpleTransform()", tr.BasicSimpleTransform.__init__, lambda r: r.transforms.BasicSimpleTransform.__init__),
        ("Basic.get_heat_map", tr.BasicSimpleTransform.get_heat_map, lambda r: r.transforms.BasicSimpleTransform.get_heat_map),
        ("box_to_center_scale", ju.box_to_center_scale, lambda r: r.joint_utils.box_to_center_scale),
        ("center_scale_to_box", ju.center_scale_to_box, lambda r: r.joint_utils.center_scale_to_box),
        ("get_affine_transform", ju.get_affine_transform, lambda r: r.joint_utils.get_affine_transform),
        ("affine_transform_batch", ju.affine_transform_batch, lambda r: r.joint_utils.affine_transform_batch),
        ("flip_joints", ju.flip_joints, lambda r: r.joint_utils.flip_joints),
        ("oks_iou", nd.oks_iou, lambda r: r.naive_data.oks_iou),
        ("oks_nms", nd.oks_nms, lambda r: r.naive_data.oks_nms),
        ("heat_map_to_axis", pm.BasicKeyPointDecoder.heat_map_to_axis, lambda r: r.pose_metrics.BasicKeyPointDecoder.heat_map_to_axis),
        ("BasicKeyPointDecoder.__call__", pm.BasicKeyPointDecoder.__call__, lambda r: r.pose_metrics.BasicKeyPointDecoder.__call__),
        ("GaussTaylorKeyPointDecoder()", pm.GaussTaylorKeyPointDecoder.__init__, lambda r: r.pose_metrics.GaussTaylorKeyPointDecoder.__init__),
        ("GaussTaylorKeyPointDecoder.__call__", pm.GaussTaylorKeyPointDecoder.__call__,
         lambda r: r.pose_metrics.GaussTaylorKeyPointDecoder.__call__),
        ("DarkPoseOriginalKeyPointDecoder()", pm.DarkPoseOriginalKeyPointDecoder.__init__,
         lambda r: r.pose_metrics.DarkPoseOriginalKeyPointDecoder.__init__),
        ("DarkPoseOriginal.__call__", pm.DarkPoseOriginalKeyPointDecoder.__call__, lambda r: r.pose_metrics.DarkPoseOriginalKeyPointDecoder.__call__),
        ("HeatMapAcc()", pm.HeatMapAcc.__init__, lambda r: r.pose_metrics.HeatMapAcc.__init__),
        ("HeatMapAcc.__call__", pm.HeatMapAcc.__call__, lambda r: r.pose_metrics.HeatMapAcc.__call__),
        ("kps_to_dict_", pm.kps_to_dict_, lambda r: r.pose_metrics.kps_to_dict_),
    ]


def _recordable(fn):
    """Parameter list as JSON: [name, repr of the default or None when there is none]."""
    return [[n, None if d is inspect.Parameter.empty else repr(d)] for n, d in _params(fn)]


def test_mirrored_signatures():
    ref = ref_loader.load() if ref_loader.available() else None
    with open(RECORD) as fh:
        record = json.load(fh)
    add_missing = os.environ.get("SP_RECORD_REFERENCE_PINS") == "missing"
    for label, our_fn, ref_fn in _mirrored():
        if ref is not None:
            _check(ref_fn(ref), our_fn, label)
        ours = _recordable(our_fn)
        if label not in record and add_missing:
            record[label] = ours
            continue
        want = record[label]
        assert ours[:len(want)] == want, (label, want, ours)
        for name, default in ours[len(want):]:
            assert default is not None, (label, "extra parameter without default", name)
    if add_missing:
        with open(RECORD, "w") as fh:
            json.dump(record, fh, indent=1, sort_keys=True)
            fh.write("\n")
    from simple_pose_b200.metrics import pose_metrics as pm
    from simple_pose_b200.commons import transforms as tr
    # class relationships the reference's code relies on (HeatMapAcc calls heat_map_to_axis on the class)
    assert issubclass(pm.GaussTaylorKeyPointDecoder, pm.BasicKeyPointDecoder)
    assert isinstance(inspect.getattr_static(pm.BasicKeyPointDecoder, "heat_map_to_axis"), staticmethod)
    assert isinstance(inspect.getattr_static(tr.RefineSimpleTransform, "get_heat_map"), staticmethod)
