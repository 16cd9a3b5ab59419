"""CPU: the oracle (and the host-side mirror of the head) against the reference's OWN source.

The reference's outputs on the inputs built below were recorded by executing its code in place through
oracle/ref_shim.py (tests/golden/make_golden.py, which calls the builders of this module) and are stored in
tests/golden/oracle_vs_reference.npz, so these tests need no reference checkout.  Inputs are regenerated from
their seeds; a fingerprint of each is stored next to the outputs, so a changed input generator fails loudly
instead of looking like a numerical mismatch.  Outputs too large to store whole are kept as a sketch: a fixed
sample of entries, the row sums and the Frobenius norm (sketch())."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from balancedgroupsoftmax_b200.tables import synthetic_tables, load_reference_files, save_reference_files
from oracle import bags_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'oracle_vs_reference.npz')

LOSS_CASES = [(1, 1, 0), (1, 0, 1), (64, 16, 2), (300, 75, 3), (512, 128, 4), (40, 40, 5)]
REWEIGHT_CASES = [(300, 75, 1), (64, 0, 2), (40, 40, 3), (512, 128, 4)]
NMS_CONFIGS = [(0.05, 0.5, 20), (0.0, 0.3, 1000), (0.9999, 0.5, 10), (0.2, 0.5, -1)]
BBOX_MEANS, BBOX_STDS = [0., 0., 0., 0.], [0.1, 0.1, 0.2, 0.2]

SKETCH_SAMPLE = 1024
SKETCH_STRIDE = 7919    # prime, so the sampled flat indices are distinct for every array size sketched here


# ------------------------------------------------------------------------------------------------ inputs
def tables():
    return synthetic_tables(1231, seed=0)


# Normal draws come from numpy's RandomState: torch's CPU normal sampler gives different numbers on different
# vector instruction sets, and these inputs must match the ones the reference outputs were recorded on.
def normal(rng, std, *shape):
    return torch.from_numpy(rng.normal(0.0, std, shape).astype(np.float32))


def head_inputs(t, N, npos, seed, K):
    """fc_cls weight ~ N(0, 0.2), bias ~ N(0, 0.1), ReLU features, the first npos RoIs foreground."""
    rng = np.random.RandomState(seed)
    W = normal(rng, 0.2, t.num_logits, K)
    b = normal(rng, 0.1, t.num_logits)
    x = torch.relu(normal(rng, 1.0, N, K))
    labels = torch.zeros(N, dtype=torch.long)
    labels[:npos] = torch.from_numpy(rng.randint(1, t.num_classes, npos).astype(np.int64))
    return x, W, b, labels


def merge_inputs(t):
    rng = np.random.RandomState(7)
    return [normal(rng, 3.0, 200, t.num_logits) for _ in range(3)]


def sampler_labels():
    labels = torch.zeros(400, dtype=torch.long)
    labels[:90] = torch.randint(1, 1231, (90,), generator=torch.Generator().manual_seed(3))
    return labels


def bbox_target_inputs():
    """Four images: positives and negatives, negatives only, positives only, one of each."""
    g = torch.Generator().manual_seed(11)

    def boxes(n):
        xy = torch.rand(n, 2, generator=g) * 600
        wh = torch.rand(n, 2, generator=g) * 200 + 1
        return torch.cat([xy, xy + wh], 1)

    imgs = []
    for npos, nneg in ((5, 20), (0, 12), (7, 0), (1, 1)):
        imgs.append(SimpleNamespace(pos_bboxes=boxes(npos), neg_bboxes=boxes(nneg), pos_gt_bboxes=boxes(npos),
                                    pos_gt_labels=torch.randint(1, 1231, (npos,), generator=g)))
    return imgs


class ConfigDict(dict):
    """Stand-in for mmcv.ConfigDict (attribute access on dict keys), the type of the reference's train config."""
    __getattr__ = dict.__getitem__


def bbox_target_args(imgs, pos_weight):
    return ([r.pos_bboxes for r in imgs], [r.neg_bboxes for r in imgs], [r.pos_gt_bboxes for r in imgs],
            [r.pos_gt_labels for r in imgs], ConfigDict(pos_weight=pos_weight))


def nms_inputs():
    """60 boxes, 9 classes; class-agnostic boxes and per-class boxes."""
    g = torch.Generator().manual_seed(5)
    n, classes = 60, 9
    xy = torch.rand(n, 2, generator=g) * 80
    wh = torch.rand(n, 2, generator=g) * 40 + 2
    boxes4 = torch.cat([xy, xy + wh], 1)
    boxes_pc = (boxes4[:, None, :] + torch.rand(n, classes, 4, generator=g)).reshape(n, classes * 4)
    scores = torch.rand(n, classes, generator=g) ** 3
    return [boxes4, boxes_pc], scores


def reweight_class_weights(t):
    g = torch.Generator().manual_seed(21)
    return [torch.rand(int(t.pred_slice[b, 1]), generator=g) * 2 + 0.1 for b in range(1, t.num_bins)]


def fingerprint(*tensors):
    """Sum and sum of squares of every input, in float64."""
    return np.array([v for a in tensors for v in (a.double().sum().item(), a.double().pow(2).sum().item())])


def sketch(a):
    """A fixed sample of the entries, the row sums and the Frobenius norm of a 2-D array."""
    a = np.asarray(a, dtype=np.float64)
    flat = a.reshape(-1)
    idx = np.arange(min(SKETCH_SAMPLE, flat.size)) * SKETCH_STRIDE % flat.size
    return {'sample': flat[idx].astype(np.float32), 'rowsum': a.sum(1).astype(np.float32),
            'norm': np.float64(np.linalg.norm(flat))}


# ------------------------------------------------------------------------------------------------ checks
@pytest.fixture(scope='module')
def ref():
    with np.load(GOLDEN) as d:
        return {k: d[k] for k in d.files}


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-20)


def check_sketch(ref, key, a, tol):
    s = sketch(a)
    for part in ('sample', 'rowsum', 'norm'):
        assert rel(s[part], ref['%s_%s' % (key, part)]) <= tol, (key, part)


def check_fingerprint(ref, key, *tensors):
    assert np.allclose(fingerprint(*tensors), ref[key + '_inputs'], rtol=1e-12, atol=0), 'inputs changed: ' + key


@pytest.mark.parametrize('N,npos,seed', LOSS_CASES)
def test_loss_and_grads_match_reference(ref, N, npos, seed):
    t = tables()
    l2b, ps = torch.from_numpy(t.label2binlabel), torch.from_numpy(t.pred_slice)
    x, W, b, labels = head_inputs(t, N, npos, seed, K=128)
    key = 'loss_n%d_p%d_s%d' % (N, npos, seed)
    check_fingerprint(ref, key, x, W, b, labels)
    np.random.seed(seed)   # the seed the reference's sampler ran with => identical sampled masks
    lo, dW, db, dX = O.head_step(x, W, b, labels, l2b, ps, 8.0)
    want = ref[key + '_losses']
    assert sorted(lo) == ['loss_cls_bin%d' % g for g in range(5)]
    for g in range(5):
        assert abs(lo['loss_cls_bin%d' % g].item() - want[g]) <= 1e-6 * max(1.0, abs(want[g])), g
    assert rel(db.numpy(), ref[key + '_db']) < 1e-6
    check_sketch(ref, key + '_dW', dW.numpy(), 1e-6)
    check_sketch(ref, key + '_dX', dX.numpy(), 1e-6)


def test_merge_score_matches_reference(ref):
    t = tables()
    ps = torch.from_numpy(t.pred_slice)
    for i, z in enumerate(merge_inputs(t)):
        check_fingerprint(ref, 'merge%d' % i, z)
        m = O.merge_score(z, ps, [torch.from_numpy(s) for s in t.fg_splits], t.num_classes)
        assert tuple(m.shape) == tuple(ref['merge%d_shape' % i])
        # bit-exact on the machine that recorded it; elsewhere the softmax's exp rounds per CPU instruction set
        check_sketch(ref, 'merge%d' % i, m.numpy(), 1e-6)
        assert np.array_equal(m.argmax(1).numpy(), ref['merge%d_argmax' % i])


def test_tables_load_into_reference_head(ref, tmp_path):
    """Files written by tables.save_reference_files hold what the reference's constructor read from them
    (gs_bbox_head_with0.py:37-49): label2binlabel, pred_slice and the four foreground splits."""
    t = tables()
    back = load_reference_files(**save_reference_files(t, str(tmp_path)))
    for tab in (t, back):
        assert tab.label2binlabel.dtype == np.int64 and tab.label2binlabel.shape == (5, 1231)
        assert np.array_equal(tab.label2binlabel, ref['tables_label2binlabel'])
        assert np.array_equal(tab.pred_slice, ref['tables_pred_slice'])
        assert [len(s) for s in tab.fg_splits] == ref['tables_fg_split_lens'].tolist()
        assert np.array_equal(np.concatenate(tab.fg_splits), ref['tables_fg_splits'])
        assert tab.num_logits == int(ref['tables_fc_cls_out_features']) == 1236


def test_host_mirror_numpy_sampler_is_the_reference_sampler(ref):
    """GSBBoxHeadWith0(sampler='numpy')._sample_others_numpy draws the same masks as the reference."""
    from balancedgroupsoftmax_b200.head import GSBBoxHeadWith0
    t = tables()
    mine = GSBBoxHeadWith0(num_fcs=2, in_channels=4, fc_out_channels=128, roi_feat_size=2, num_classes=1231,
                           gs_config=dict(tables=t, others_sample_ratio=8.0, num_bins=5, sampler='numpy',
                                          loss_bin=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0)))
    labels = sampler_labels()
    check_fingerprint(ref, 'sampler', labels)
    np.random.seed(11)
    for g in range(1, 5):
        w = mine._sample_others_numpy(mine.label2binlabel[g][labels])
        assert str(w.dtype) == str(ref['sampler_dtype'])
        assert np.array_equal(w.numpy(), ref['sampler_w'][g])


def test_get_target_matches_reference_bbox_target(ref):
    """The head's standalone target generator against the reference's bbox_target.py / transforms.py."""
    from balancedgroupsoftmax_b200.head import GSBBoxHeadWith0, bbox2delta, bbox_target
    imgs = bbox_target_inputs()
    check_fingerprint(ref, 'bbox', *[a for r in imgs for a in vars(r).values()])

    def same(got, key):
        assert str(got.dtype) == str(ref[key + '_dtype']), key
        assert np.array_equal(got.numpy(), ref[key]), key

    same(bbox2delta(imgs[0].pos_bboxes, imgs[0].pos_gt_bboxes, BBOX_MEANS, BBOX_STDS), 'bbox2delta')
    for pos_weight in (-1, 2.5):
        args = bbox_target_args(imgs, pos_weight)
        got = bbox_target(*args, reg_classes=1231, target_means=BBOX_MEANS, target_stds=BBOX_STDS)
        assert len(got) == 4
        for j, a in enumerate(got):
            same(a, 'bbox_pw%g_%d' % (pos_weight, j))
        # not concatenated
        got = bbox_target(*args, target_means=BBOX_MEANS, target_stds=BBOX_STDS, concat=False)
        assert len(got) == 4
        for j, la in enumerate(got):
            assert len(la) == len(imgs)
            for i, a in enumerate(la):
                same(a, 'bbox_pw%g_split%d_%d' % (pos_weight, j, i))
    # through the head method
    t = tables()
    head = GSBBoxHeadWith0(num_fcs=1, in_channels=4, fc_out_channels=16, roi_feat_size=1, num_classes=t.num_classes,
                           target_means=BBOX_MEANS, target_stds=BBOX_STDS,
                           gs_config=dict(tables=t, others_sample_ratio=8.0, num_bins=5,
                                          loss_bin=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0)))
    got = head.get_target(imgs, None, None, ConfigDict(pos_weight=-1))
    assert len(got) == 4
    for j, a in enumerate(got):
        same(a, 'bbox_pw-1_%d' % j)
    assert got[0].dtype == torch.long and got[0][:5].tolist() == imgs[0].pos_gt_labels.tolist() and got[0][5:25].sum() == 0


def test_multiclass_nms_oracle_matches_reference_loop(ref):
    """The oracle's multiclass_nms against the reference's bbox_nms.py loop (its compiled NMS op replaced by the
    oracle's greedy "+1" NMS when the outputs were recorded): thresholds, labels, class order and the top-k rule."""
    boxes, scores = nms_inputs()
    check_fingerprint(ref, 'nms', *boxes, scores)
    for bi, mb in enumerate(boxes):
        for ci, (thr, iou, k) in enumerate(NMS_CONFIGS):
            got = O.multiclass_nms(mb, scores.clone(), thr, iou, k)
            key = 'nms_b%d_c%d' % (bi, ci)
            assert str(got[0].dtype) == str(ref[key + '_dtype']) and str(got[1].dtype) == str(ref[key + '_labels_dtype'])
            assert np.array_equal(got[0].numpy(), ref[key + '_dets']) and np.array_equal(got[1].numpy(), ref[key + '_labels'])


def test_reweight_variant_matches_reference(ref):
    """Reweight head variant (gs_bbox_head_with0_reweight.py): the oracle's weights / normalisers / per-bin losses
    against the reference class."""
    t = tables()
    cls_weights = reweight_class_weights(t)
    check_fingerprint(ref, 'reweight_cls', *cls_weights)
    l2b, ps = torch.from_numpy(t.label2binlabel), torch.from_numpy(t.pred_slice)
    for N, npos, seed in REWEIGHT_CASES:
        x, W, b, labels = head_inputs(t, N, npos, seed, K=64)
        key = 'reweight_n%d_p%d_s%d' % (N, npos, seed)
        check_fingerprint(ref, key, x, W, b, labels)
        z = O.fc_cls(x, W, b)
        np.random.seed(seed)
        remapped = O.remap_labels_reweight(labels, l2b, 8.0, cls_weights)
        for g, a in enumerate(remapped[1]):
            assert np.array_equal(a.float().numpy(), ref[key + '_weights'][g])
        assert [float(a) for a in remapped[2]] == ref[key + '_avg'].tolist()
        got = O.bags_loss(z, labels, l2b, ps, remapped=remapped)
        want = ref[key + '_losses']
        for g in range(5):
            v = got['loss_cls_bin%d' % g].item()
            assert abs(v - want[g]) <= 1e-6 * max(1.0, abs(want[g])), (g, v, want[g])
