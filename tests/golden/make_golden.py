"""Generate tests/golden/*.npz by executing the REFERENCE'S OWN source (through
oracle/ref_shim.py) on CPU, with $BAGS_REFERENCE_DIR pointing at a reference checkout:

    python tests/golden/make_golden.py [NAME ...]      (default: every fixture)

The reference ships no golden vectors for this path (SURVEY.md §4/§8c); these fixtures are the
pinning: inputs + the reference's outputs (per-bin losses, sampled masks, avg factors, grads,
merged scores).  With them the tests run without a reference checkout.

Fixture shapes are small on the K (feature) axis so the files stay tiny; the logit axis keeps
the full 1236-wide, 5-bin structure.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from balancedgroupsoftmax_b200.tables import synthetic_tables  # noqa: E402
from oracle import ref_shim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def make_case(name, N, K, npos, seed, wstd, ratio=8.0, gout=None, zipf=False):
    tables = synthetic_tables(1231, seed=0)
    head = ref_shim.build_reference_head(tables, others_sample_ratio=ratio, fc_out_channels=K)
    torch.manual_seed(seed)
    np.random.seed(seed)
    with torch.no_grad():
        head.fc_cls.weight.normal_(0, wstd)
        head.fc_cls.bias.normal_(0, 0.1)
    x = torch.relu(torch.randn(N, K))
    labels = torch.zeros(N, dtype=torch.long)
    if npos > 0:
        if zipf:
            r = np.random.zipf(1.3, size=npos)
            labels[:npos] = torch.from_numpy(((r - 1) % 1230) + 1)
        else:
            labels[:npos] = torch.randint(1, 1231, (npos,))
    rec = {}
    orig = head._remap_labels

    def wrap(l):
        r = orig(l)
        rec['r'] = r
        return r

    head._remap_labels = wrap
    xr = x.clone().requires_grad_(True)
    z = head.fc_cls(xr)
    losses = head.loss(z, None, labels, None, None, None)
    g = [1.0] * 5 if gout is None else gout
    total = sum(gi * losses['loss_cls_bin%d' % i] for i, gi in enumerate(g))
    total.backward()
    merged = head._merge_score(z.detach())
    new_labels, new_weights, new_avg = rec['r']
    np.savez_compressed(
        os.path.join(OUT, name + '.npz'),
        x=x.numpy(), weight=head.fc_cls.weight.detach().numpy(), bias=head.fc_cls.bias.detach().numpy(),
        labels=labels.numpy(), ratio=np.float64(ratio), gout=np.asarray(g, dtype=np.float32),
        logits_sample=z.detach()[:, ::29].numpy(),
        losses=np.asarray([losses['loss_cls_bin%d' % i].item() for i in range(5)], dtype=np.float64),
        bin_labels=np.stack([t.numpy() for t in new_labels]).astype(np.int16),
        wmask=np.stack([w.numpy() for w in new_weights]).astype(np.uint8),
        avg=np.asarray(new_avg, dtype=np.float64),
        dW=head.fc_cls.weight.grad.numpy(), db=head.fc_cls.bias.grad.numpy(), dX=xr.grad.numpy(),
        merged_argmax=merged.argmax(1).numpy().astype(np.int16),
        merged_fg_argmax=(merged[:, 1:].argmax(1) + 1).numpy().astype(np.int16),
        merged_rowsum=merged.sum(1).numpy(), merged_sample=merged[:, ::37].numpy(),
        seed=np.int64(seed),
    )
    print(name, 'losses', [round(losses['loss_cls_bin%d' % i].item(), 5) for i in range(5)], 'avg', new_avg)


def make_oracle_vs_reference():
    """The reference's outputs on the inputs of tests/test_oracle_vs_reference.py (built by that module)."""
    import test_oracle_vs_reference as T
    from oracle import bags_oracle as O
    out = {}

    def put_sketch(key, a):
        for part, v in T.sketch(a).items():
            out['%s_%s' % (key, part)] = v

    t = T.tables()
    head = ref_shim.build_reference_head(t, fc_out_channels=128)
    head.init_weights()
    for N, npos, seed in T.LOSS_CASES:
        x, W, b, labels = T.head_inputs(t, N, npos, seed, K=128)
        key = 'loss_n%d_p%d_s%d' % (N, npos, seed)
        out[key + '_inputs'] = T.fingerprint(x, W, b, labels)
        with torch.no_grad():
            head.fc_cls.weight.copy_(W)
            head.fc_cls.bias.copy_(b)
        np.random.seed(seed)
        xr = x.clone().requires_grad_(True)
        head.zero_grad()
        losses = head.loss(head.fc_cls(xr), None, labels, None, None, None)
        sum(losses.values()).backward()
        assert set(losses) == {'loss_cls_bin%d' % g for g in range(5)}
        out[key + '_losses'] = np.array([losses['loss_cls_bin%d' % g].item() for g in range(5)])
        out[key + '_db'] = head.fc_cls.bias.grad.numpy()
        put_sketch(key + '_dW', head.fc_cls.weight.grad.numpy())
        put_sketch(key + '_dX', xr.grad.numpy())

    for i, z in enumerate(T.merge_inputs(t)):
        m = head._merge_score(z)
        out['merge%d_inputs' % i] = T.fingerprint(z)
        out['merge%d_shape' % i] = np.array(m.shape)
        out['merge%d_argmax' % i] = m.argmax(1).numpy()
        put_sketch('merge%d' % i, m.numpy())

    out['tables_label2binlabel'] = head.label2binlabel.numpy()
    out['tables_pred_slice'] = head.pred_slice.numpy()
    out['tables_fg_split_lens'] = np.array([len(s) for s in head.fg_splits])
    out['tables_fg_splits'] = torch.cat(head.fg_splits).numpy()
    out['tables_fc_cls_out_features'] = np.int64(head.fc_cls.out_features)

    labels = T.sampler_labels()
    out['sampler_inputs'] = T.fingerprint(labels)
    np.random.seed(11)
    _, ref_w, _ = head._remap_labels(labels)
    out['sampler_w'] = torch.stack(ref_w).numpy()
    out['sampler_dtype'] = np.str_(ref_w[1].dtype)

    def put_exact(key, a):
        out[key] = a.numpy()
        out[key + '_dtype'] = np.str_(a.dtype)

    ref_bbox_target, ref_bbox2delta = ref_shim.load_bbox_target()
    imgs = T.bbox_target_inputs()
    out['bbox_inputs'] = T.fingerprint(*[a for r in imgs for a in vars(r).values()])
    put_exact('bbox2delta', ref_bbox2delta(imgs[0].pos_bboxes, imgs[0].pos_gt_bboxes, T.BBOX_MEANS, T.BBOX_STDS))
    for pos_weight in (-1, 2.5):
        args = T.bbox_target_args(imgs, pos_weight)
        for j, a in enumerate(ref_bbox_target(*args, reg_classes=1231, target_means=T.BBOX_MEANS,
                                              target_stds=T.BBOX_STDS)):
            put_exact('bbox_pw%g_%d' % (pos_weight, j), a)
        for j, la in enumerate(ref_bbox_target(*args, target_means=T.BBOX_MEANS, target_stds=T.BBOX_STDS,
                                               concat=False)):
            for i, a in enumerate(la):
                put_exact('bbox_pw%g_split%d_%d' % (pos_weight, j, i), a)

    ref_mc_nms = ref_shim.load_multiclass_nms(O.nms_plus1)
    boxes, scores = T.nms_inputs()
    out['nms_inputs'] = T.fingerprint(*boxes, scores)
    for bi, mb in enumerate(boxes):
        for ci, (thr, iou, k) in enumerate(T.NMS_CONFIGS):
            dets, lab = ref_mc_nms(mb, scores.clone(), thr, dict(type='nms', iou_thr=iou), k)
            key = 'nms_b%d_c%d' % (bi, ci)
            out[key + '_dets'], out[key + '_dtype'] = dets.numpy(), np.str_(dets.dtype)
            out[key + '_labels'], out[key + '_labels_dtype'] = lab.numpy(), np.str_(lab.dtype)

    cls_weights = T.reweight_class_weights(t)
    out['reweight_cls_inputs'] = T.fingerprint(*cls_weights)
    head = ref_shim.build_reference_reweight_head(t, cls_weights, fc_out_channels=64)
    head.init_weights()
    for N, npos, seed in T.REWEIGHT_CASES:
        x, W, b, labels = T.head_inputs(t, N, npos, seed, K=64)
        key = 'reweight_n%d_p%d_s%d' % (N, npos, seed)
        out[key + '_inputs'] = T.fingerprint(x, W, b, labels)
        with torch.no_grad():
            head.fc_cls.weight.copy_(W)
            head.fc_cls.bias.copy_(b)
            z = head.fc_cls(x)
        np.random.seed(seed)
        losses = head.loss(z, None, labels, None, None, None)
        out[key + '_losses'] = np.array([losses['loss_cls_bin%d' % g].item() for g in range(5)])
        np.random.seed(seed)
        _, rw, ra = head._remap_labels(labels)
        out[key + '_weights'] = torch.stack([w.float() for w in rw]).numpy()
        out[key + '_avg'] = np.array([float(a) for a in ra])
    np.savez_compressed(os.path.join(OUT, 'oracle_vs_reference.npz'), **out)
    print('oracle_vs_reference', len(out), 'arrays')


def make_weighted_loss_kat():
    # known-answer numbers of the weighted_loss doctest (mmdet/models/losses/utils.py:66-83), evaluated by
    # the reference's own decorator
    ns = ref_shim.load()

    @ns.weighted_loss
    def l1_loss(pred, target):
        return (pred - target).abs()

    pred, target, weight = torch.Tensor([0, 2, 3]), torch.Tensor([1, 1, 1]), torch.Tensor([1, 0, 1])
    np.savez(os.path.join(OUT, 'weighted_loss_kat.npz'),
             mean=l1_loss(pred, target).item(), weighted=l1_loss(pred, target, weight).item(),
             none=l1_loss(pred, target, reduction='none').numpy(),
             avg2=l1_loss(pred, target, weight, avg_factor=2).item())


FIXTURES = {
    'ref_n96_k64': lambda: make_case('ref_n96_k64', N=96, K=64, npos=24, seed=1, wstd=0.3),
    'ref_n257_k64_cascade': lambda: make_case('ref_n257_k64_cascade', N=257, K=64, npos=70, seed=2, wstd=0.2,
                                              gout=[1.0, 0.5, 0.25, 0.5, 1.0]),
    'ref_n64_k32_allbg': lambda: make_case('ref_n64_k32_allbg', N=64, K=32, npos=0, seed=3, wstd=0.3),
    'ref_n48_k32_allfg': lambda: make_case('ref_n48_k32_allfg', N=48, K=32, npos=48, seed=4, wstd=0.3, zipf=True),
    'weighted_loss_kat': make_weighted_loss_kat,
    'oracle_vs_reference': make_oracle_vs_reference,
}


if __name__ == '__main__':
    assert ref_shim.available(), 'reference checkout not reachable (set $BAGS_REFERENCE_DIR)'
    for name in sys.argv[1:] or list(FIXTURES):
        FIXTURES[name]()
