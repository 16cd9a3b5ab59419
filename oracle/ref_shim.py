"""Execute the reference's OWN hot-path source on CPU, in place -- TEST INFRASTRUCTURE.

The reference (FishYuLi/BalancedGroupSoftmax) cannot be installed here (needs
mmcv, pycocotools and THC-era CUDA extensions), but the files on the hot path
are plain PyTorch.  This shim loads them straight from a reference checkout
(``$BAGS_REFERENCE_DIR`` or ``baseline/_ref``) with
importlib, stubbing only what they import from outside the path (mmcv.is_str,
mmdet.core.{bbox_target,delta2bbox,multiclass_nms}, ConvModule) and making
``Tensor.cuda()`` the identity so the head builds on CPU.  Nothing is copied
into this repository.

Used by tests/golden/make_golden.py (the reference outputs the tests compare
against) and by the CPU arm of bench.py; never by the product.  ``available()``
is False where no checkout is configured.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import tempfile
import types
from typing import Optional

_CANDIDATES = [os.environ.get('BAGS_REFERENCE_DIR', ''),
               os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'baseline', '_ref')]

_loaded = None


def reference_dir() -> Optional[str]:
    for c in _CANDIDATES:
        if c and os.path.isfile(os.path.join(c, 'mmdet', 'models', 'bbox_heads', 'gs_bbox_head_with0.py')):
            return c
    return None


def available() -> bool:
    return reference_dir() is not None


def _shell(name: str, path: str) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__path__ = [path]
    sys.modules[name] = m
    return m


def _exec(name: str, file: str) -> types.ModuleType:
    spec = importlib.util.spec_from_file_location(name, file)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


class AttrDict(dict):
    """Stand-in for mmcv.ConfigDict (attribute access on dict keys)."""
    __getattr__ = dict.__getitem__


def load():
    """Returns a namespace with GSBBoxHeadWith0, CrossEntropyLoss, weighted_loss, ... of the reference."""
    global _loaded
    if _loaded is not None:
        return _loaded
    root = reference_dir()
    if root is None:
        raise RuntimeError('reference checkout not reachable')
    import torch

    if 'mmcv' not in sys.modules:
        mmcv = types.ModuleType('mmcv')
        mmcv.is_str = lambda x: isinstance(x, str)
        sys.modules['mmcv'] = mmcv
    md = os.path.join(root, 'mmdet')
    _shell('mmdet', md)
    utils = _shell('mmdet.utils', os.path.join(md, 'utils'))
    _shell('mmdet.models', os.path.join(md, 'models'))
    _shell('mmdet.models.bbox_heads', os.path.join(md, 'models', 'bbox_heads'))
    losses = _shell('mmdet.models.losses', os.path.join(md, 'models', 'losses'))
    mutils = _shell('mmdet.models.utils', os.path.join(md, 'models', 'utils'))
    core = _shell('mmdet.core', os.path.join(md, 'core'))
    _shell('mmdet.core.fp16', os.path.join(md, 'core', 'fp16'))

    reg = _exec('mmdet.utils.registry', os.path.join(md, 'utils', 'registry.py'))
    utils.Registry, utils.build_from_cfg = reg.Registry, reg.build_from_cfg
    _exec('mmdet.models.registry', os.path.join(md, 'models', 'registry.py'))
    _exec('mmdet.models.builder', os.path.join(md, 'models', 'builder.py'))
    _exec('mmdet.core.fp16.utils', os.path.join(md, 'core', 'fp16', 'utils.py'))
    dec = _exec('mmdet.core.fp16.decorators', os.path.join(md, 'core', 'fp16', 'decorators.py'))
    core.auto_fp16, core.force_fp32 = dec.auto_fp16, dec.force_fp32
    core.bbox_target = core.delta2bbox = core.multiclass_nms = None
    lutils = _exec('mmdet.models.losses.utils', os.path.join(md, 'models', 'losses', 'utils.py'))
    ce = _exec('mmdet.models.losses.cross_entropy_loss', os.path.join(md, 'models', 'losses', 'cross_entropy_loss.py'))
    sl1 = _exec('mmdet.models.losses.smooth_l1_loss', os.path.join(md, 'models', 'losses', 'smooth_l1_loss.py'))
    acc = _exec('mmdet.models.losses.accuracy', os.path.join(md, 'models', 'losses', 'accuracy.py'))
    losses.accuracy = acc.accuracy
    mutils.ConvModule = None
    _exec('mmdet.models.bbox_heads.bbox_head', os.path.join(md, 'models', 'bbox_heads', 'bbox_head.py'))
    _exec('mmdet.models.bbox_heads.convfc_bbox_head', os.path.join(md, 'models', 'bbox_heads', 'convfc_bbox_head.py'))
    gs = _exec('mmdet.models.bbox_heads.gs_bbox_head_with0',
               os.path.join(md, 'models', 'bbox_heads', 'gs_bbox_head_with0.py'))

    # the head calls .cuda() on its tables and sampled indices (gs_bbox_head_with0.py:37-49,85,255-256)
    torch.Tensor.cuda = lambda self, *a, **k: self

    ns = types.SimpleNamespace(
        root=root, GSBBoxHeadWith0=gs.GSBBoxHeadWith0, CrossEntropyLoss=ce.CrossEntropyLoss,
        SmoothL1Loss=sl1.SmoothL1Loss, weighted_loss=lutils.weighted_loss,
        weight_reduce_loss=lutils.weight_reduce_loss, Registry=reg.Registry,
        build_from_cfg=reg.build_from_cfg, AttrDict=AttrDict)
    _loaded = ns
    return ns


def build_reference_reweight_head(tables, cls_weights, others_sample_ratio: float = 8.0, fc_out_channels: int = 1024,
                                  tmpdir: Optional[str] = None):
    """The reference's GSBBoxHeadWith0Reweight (mmdet/models/bbox_heads/gs_bbox_head_with0_reweight.py) on CPU, its
    per-bin class weights written to a pickle like the file its config names (``bin_cls_weight``)."""
    import pickle
    import numpy as np
    from balancedgroupsoftmax_b200.tables import save_reference_files
    load()
    root = reference_dir()
    md = os.path.join(root, 'mmdet')
    # this repository's drop-in registers itself under the same name when an `mmdet` package is importable
    sys.modules['mmdet.models.registry'].HEADS._module_dict.pop('GSBBoxHeadWith0Reweight', None)
    mod = _exec('mmdet.models.bbox_heads.gs_bbox_head_with0_reweight',
                os.path.join(md, 'models', 'bbox_heads', 'gs_bbox_head_with0_reweight.py'))
    d = tmpdir or tempfile.mkdtemp(prefix='bags_tables_rw_')
    paths = save_reference_files(tables, d)
    wpath = os.path.join(d, 'bin_cls_weight.pkl')
    with open(wpath, 'wb') as f:
        pickle.dump([np.asarray(w, dtype=np.float32) for w in cls_weights], f)
    gs_config = AttrDict(
        label2binlabel=paths['label2binlabel'], pred_slice=paths['pred_slice'], fg_split=paths['fg_split'],
        others_sample_ratio=others_sample_ratio, bin_cls_weight=wpath,
        loss_bg=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0), num_bins=tables.num_bins,
        loss_bin=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0))
    return mod.GSBBoxHeadWith0Reweight(
        num_fcs=2, in_channels=256, fc_out_channels=fc_out_channels, gs_config=gs_config, roi_feat_size=7,
        num_classes=tables.num_classes, target_means=[0., 0., 0., 0.], target_stds=[0.1, 0.1, 0.2, 0.2],
        reg_class_agnostic=False, loss_cls=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0),
        loss_bbox=dict(type='SmoothL1Loss', beta=1.0, loss_weight=1.0))


def load_bbox_target():
    """The reference's own ``bbox_target`` (mmdet/core/bbox/bbox_target.py) and ``bbox2delta`` (transforms.py),
    executed in place: the producer of the head's ``labels`` / box targets."""
    load()
    root = reference_dir()
    md = os.path.join(root, 'mmdet')
    import functools
    if 'mmdet.core.utils' not in sys.modules or not hasattr(sys.modules['mmdet.core.utils'], 'multi_apply'):
        cu = _shell('mmdet.core.utils', os.path.join(md, 'core', 'utils'))

        def multi_apply(func, *args, **kwargs):   # mmdet/core/utils/misc.py:22-25 (its module imports six / mmcv.im*)
            pfunc = functools.partial(func, **kwargs) if kwargs else func
            return tuple(map(list, zip(*map(pfunc, *args))))
        cu.multi_apply = multi_apply
    _shell('mmdet.core.bbox', os.path.join(md, 'core', 'bbox'))
    tr = _exec('mmdet.core.bbox.transforms', os.path.join(md, 'core', 'bbox', 'transforms.py'))
    bt = _exec('mmdet.core.bbox.bbox_target', os.path.join(md, 'core', 'bbox', 'bbox_target.py'))
    return bt.bbox_target, tr.bbox2delta


def load_multiclass_nms(nms_op):
    """The reference's own ``multiclass_nms`` loop (mmdet/core/post_processing/bbox_nms.py) executed in place, with
    ``nms_op(dets, iou_thr) -> (dets, inds)`` standing in for its compiled NMS extension (mmdet/ops/nms)."""
    load()
    root = reference_dir()
    md = os.path.join(root, 'mmdet')
    _shell('mmdet.ops', os.path.join(md, 'ops'))
    nms_pkg = _shell('mmdet.ops.nms', os.path.join(md, 'ops', 'nms'))
    wrapper = types.ModuleType('mmdet.ops.nms.nms_wrapper')
    wrapper.nms = nms_op
    sys.modules['mmdet.ops.nms.nms_wrapper'] = wrapper
    nms_pkg.nms_wrapper = wrapper
    _shell('mmdet.core.post_processing', os.path.join(md, 'core', 'post_processing'))
    mod = _exec('mmdet.core.post_processing.bbox_nms', os.path.join(md, 'core', 'post_processing', 'bbox_nms.py'))
    return mod.multiclass_nms


def build_reference_head(tables, others_sample_ratio: float = 8.0, fc_out_channels: int = 1024,
                         in_channels: int = 256, roi_feat_size: int = 7, num_fcs: int = 2,
                         reg_class_agnostic: bool = False, tmpdir: Optional[str] = None):
    """Construct the reference's GSBBoxHeadWith0 on CPU with the given GroupTables
    (written to temp files in the reference's on-disk formats)."""
    from balancedgroupsoftmax_b200.tables import save_reference_files
    ns = load()
    d = tmpdir or tempfile.mkdtemp(prefix='bags_tables_')
    paths = save_reference_files(tables, d)
    gs_config = AttrDict(
        label2binlabel=paths['label2binlabel'], pred_slice=paths['pred_slice'], fg_split=paths['fg_split'],
        others_sample_ratio=others_sample_ratio,
        loss_bg=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0),
        num_bins=tables.num_bins,
        loss_bin=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0))
    head = ns.GSBBoxHeadWith0(
        num_fcs=num_fcs, in_channels=in_channels, fc_out_channels=fc_out_channels, gs_config=gs_config,
        roi_feat_size=roi_feat_size, num_classes=tables.num_classes,
        target_means=[0., 0., 0., 0.], target_stds=[0.1, 0.1, 0.2, 0.2],
        reg_class_agnostic=reg_class_agnostic,
        loss_cls=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0),
        loss_bbox=dict(type='SmoothL1Loss', beta=1.0, loss_weight=1.0))
    return head
