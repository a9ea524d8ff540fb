# -*- coding: utf-8 -*-
"""Generates tests/golden/*.pt by running the REFERENCE's own modules (imported from /root/reference, CPU, fp32)
on the deterministic synthetic weights / inputs of tests/synth.py.  Run in the build container only
(/root/reference does not exist on the GPU box); the produced fixtures are committed.

    python tests/gen_golden.py

Import recipe (SURVEY.md 8c): stub `pycuda`, `lfd.data_pipeline` (keeping the real `Sample`), and the two native
extension modules; `nms_ext` is the reference's own CPU NMS compiled by oracle/build_ref.py; the sigmoid focal loss
has no CPU implementation in the reference (sigmoid_focal_loss_ext.cpp:32,49), so its stub is the restatement of the
.cu formulas from oracle/lfd_oracle.py (pinned against torchvision in tests/test_oracle_pins.py).
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = '/root/reference'
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import synth  # noqa: E402
from oracle import lfd_oracle as orc  # noqa: E402
from oracle import build_ref  # noqa: E402


def import_reference():
    assert os.path.isdir(REF), 'reference not mounted'
    for name in ('pycuda', 'pycuda.driver'):
        sys.modules[name] = types.ModuleType(name)
    sys.modules['pycuda'].driver = sys.modules['pycuda.driver']
    spec = importlib.util.spec_from_file_location('_ref_sample', os.path.join(REF, 'lfd/data_pipeline/dataset/sample.py'))
    smod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(smod)
    dp = types.ModuleType('lfd.data_pipeline')
    dp.__path__ = []
    ds = types.ModuleType('lfd.data_pipeline.dataset')
    ds.Sample = smod.Sample
    dp.dataset = ds
    sys.modules['lfd.data_pipeline'] = dp
    sys.modules['lfd.data_pipeline.dataset'] = ds
    build_ref.build()
    nms_ext = build_ref.load_module()
    assert nms_ext is not None
    fl = types.ModuleType('sigmoid_focal_loss_ext')
    fl.forward = lambda logits, targets, num_classes, gamma, alpha: orc.sigmoid_focal_loss_forward(logits, targets, gamma, alpha)
    fl.backward = lambda logits, targets, d, num_classes, gamma, alpha: orc.sigmoid_focal_loss_backward(logits, targets, d, gamma, alpha)
    libs_u = types.ModuleType('lfd.model.utils.libs')
    libs_u.nms_ext = nms_ext
    libs_l = types.ModuleType('lfd.model.losses.libs')
    libs_l.sigmoid_focal_loss_ext = fl
    sys.modules['lfd.model.utils.libs'] = libs_u
    sys.modules['lfd.model.utils.libs.nms_ext'] = nms_ext
    sys.modules['lfd.model.losses.libs'] = libs_l
    sys.modules['lfd.model.losses.libs.sigmoid_focal_loss_ext'] = fl
    sys.path.insert(0, REF)
    import lfd.model  # noqa: F401
    from lfd.model.backbone import LFDResNet
    from lfd.model.neck import SimpleNeck
    from lfd.model.head import LFDHead
    from lfd.model import LFD
    from lfd.model import losses
    nms_mod = sys.modules['lfd.model.utils.nms']
    # current torch rejects indexing a CPU `arange` with device indices only on GPU; on CPU the reference code runs as is
    return dict(LFDResNet=LFDResNet, SimpleNeck=SimpleNeck, LFDHead=LFDHead, LFD=LFD, losses=losses, nms_mod=nms_mod, nms_ext=nms_ext)


def build_ref_model(R, cfg):
    bb, hd, lc = cfg['backbone'], cfg['head'], cfg['lfd']
    cls_loss = R['losses'].FocalLoss(use_sigmoid=True, gamma=2.0, alpha=0.25, reduction='mean', loss_weight=1.0) \
        if hd['classification_loss_type'] == 'FocalLoss' else R['losses'].CrossEntropyLoss(reduction='mean', loss_weight=1.0)
    reg_loss = R['losses'].IoULoss(eps=1e-6, reduction='mean', loss_weight=1.0)
    backbone = R['LFDResNet'](block_mode=bb['block_mode'], stem_mode=bb['stem_mode'], body_mode=None, input_channels=3,
                              stem_channels=bb['stem_channels'], body_architecture=bb['body_architecture'],
                              body_channels=bb['body_channels'], out_indices=bb['out_indices'], frozen_stages=-1,
                              activation_cfg=dict(type='ReLU', inplace=True), norm_cfg=dict(type='BatchNorm2d'),
                              init_with_weight_file=None, norm_eval=False)
    neck = R['SimpleNeck'](num_neck_channels=128, num_input_channels_list=backbone.num_output_channels_list,
                           num_input_strides_list=backbone.num_output_strides_list, norm_cfg=dict(type='BatchNorm2d'),
                           activation_cfg=dict(type='ReLU', inplace=True))
    head = R['LFDHead'](num_classes=hd['num_classes'], num_heads=len(neck.num_output_strides_list), num_input_channels=128,
                        num_head_channels=128, num_conv_layers=2, activation_cfg=dict(type='ReLU', inplace=True),
                        norm_cfg=dict(type='GroupNorm', num_groups=16) if hd.get('norm', True) else None,
                   conv_kernel_size=hd.get('conv_kernel_size', 1), share_head_flag=hd['share_head_flag'],
                        merge_path_flag=hd['merge_path_flag'], classification_loss_type=type(cls_loss).__name__,
                        regression_loss_type=type(reg_loss).__name__)
    model = R['LFD'](backbone=backbone, neck=neck, head=head, num_classes=lc['num_classes'], regression_ranges=lc['regression_ranges'],
                     gray_range_factors=lc['gray_range_factors'], range_assign_mode=lc['range_assign_mode'],
                     point_strides=neck.num_output_strides_list, classification_loss_func=cls_loss, regression_loss_func=reg_loss,
                     distance_to_bbox_mode=lc['distance_to_bbox_mode'])
    return model


FORWARD_CASES = {  # cfg -> (N, H, W, cls_bias)
    'WIDERFACE_XS': (1, 120, 200, -1.0),
    'WIDERFACE_S': (2, 184, 248, -1.0),
    'WIDERFACE_L': (2, 160, 224, -1.0),
    'TT100K_L': (2, 136, 200, 0.0),
}
ASSIGN_CASES = {  # cfg -> (H, W) of the virtual training crop
    'WIDERFACE_S': (480, 480),
    'WIDERFACE_L': (640, 640),
    'TT100K_L': (512, 640),
}


def sizes_for(cfg, h, w):
    strides = orc.strides_of(cfg)
    taps = sorted(cfg['backbone']['out_indices'])
    stem_stride = 2 if cfg['backbone']['stem_mode'] == 'fast' else 4

    def down(v, times):
        for _ in range(times):
            v = (v + 1) // 2
        return v
    out = []
    for (s, _), st in zip(taps, strides):
        t = int(np.log2(st))
        out.append((down(h, t), down(w, t)))
    assert stem_stride in (2, 4)
    return out


def forward_case(R, name, n, h, w, cls_bias, out_dir):
    """One forward / results / loss golden of the reference model `name` on the synthetic weights and input."""
    cfg = orc.CONFIGS[name]
    model = build_ref_model(R, cfg)
    sd = synth.synth_state_dict(model.state_dict(), seed=666, cls_bias=cls_bias)
    model.load_state_dict(sd, strict=True)
    model.eval()
    x = synth.synth_input(n, h, w)
    with torch.no_grad():
        cls, reg = model(x)
    sizes = [model.head_indexes_to_feature_map_sizes[i] for i in range(len(model.head_indexes_to_feature_map_sizes))]
    assert sizes == sizes_for(cfg, h, w), (sizes, sizes_for(cfg, h, w))
    meta = [dict(resized_height=h, resized_width=w, resize_scale=1.0) for _ in range(n)]
    meta[-1]['resize_scale'] = 0.75
    results = {}
    probs = cls.sigmoid() if cfg['head']['classification_loss_type'] == 'FocalLoss' else cls.softmax(-1)[..., :-1]
    is_focal = cfg['head']['classification_loss_type'] == 'FocalLoss'
    for (thr, iou) in (((0.5, 0.3), (0.2, 0.4), (0.05, 0.4)) if is_focal else ((0.1, 0.3), (0.04, 0.4))):
        model._classification_threshold = thr
        model._nms_cfg = dict(type='nms', iou_thr=iou)
        with torch.no_grad():
            res = model.get_results((cls, reg), meta)
        results[(thr, iou)] = [torch.tensor(r, dtype=torch.float32).reshape(-1, 6) for r in res]
        print('  %s thr=%.3f iou=%.1f: pass=%d kept=%s' % (name, thr, iou, int((probs > thr).sum()), [len(r) for r in res]))
    # loss + gradients w.r.t. the outputs (annotations scaled to this small crop)
    ann = synth.synth_annotations(n, h, w, cfg['lfd']['num_classes'], seed=11, max_boxes=6)
    cls_g, reg_g = cls.clone().requires_grad_(True), reg.clone().requires_grad_(True)
    ld = model.get_loss((cls_g, reg_g), ann)
    ld['loss'].backward()
    torch.save(dict(cfg=name, N=n, H=h, W=w, cls_bias=cls_bias, seed=666, keys=[(k, tuple(v.shape)) for k, v in sd.items()],
                    checksum=synth.state_checksum(sd), sizes=sizes, cls=cls, reg=reg, meta=meta,
                    results=results, ann=ann, loss_values=ld['loss_values'], grad_cls=cls_g.grad.clone(), grad_reg=reg_g.grad.clone()),
               os.path.join(out_dir, 'forward_%s.pt' % name))
    print('forward %s: P=%d cls %s loss %s' % (name, cls.shape[1], tuple(cls.shape), ld['loss_values']))


def reference_nms_case(nms_ext, out_dir):
    """The reference's compiled CPU NMS (nms_cpu.cpp) on seeded random boxes, kept indices per (box set, IoU threshold)."""
    rng = np.random.RandomState(3)
    cases = []
    for n in (1, 7, 300):
        d = np.concatenate([rng.uniform(0, 100, (n, 2)), rng.uniform(1, 40, (n, 2)), rng.uniform(0, 1, (n, 1))], 1).astype(np.float32)
        d[:, 2:4] += d[:, 0:2]
        for thr in (0.3, 0.6):
            cases.append(dict(dets=d, thr=thr, keep=nms_ext.nms(torch.from_numpy(d), thr).numpy()))
    torch.save(cases, os.path.join(out_dir, 'reference_nms.pt'))
    print('reference nms: kept %s' % [len(c['keep']) for c in cases])


def main():
    R = import_reference()
    out_dir = os.path.join(HERE, 'golden')
    os.makedirs(out_dir, exist_ok=True)
    torch.set_num_threads(8)

    # ---- known-answer vectors from the reference docstrings, evaluated with the reference's own code
    dets = np.array([[49.1, 32.4, 51.0, 35.9, 0.9], [49.3, 32.9, 51.0, 35.3, 0.9], [49.2, 31.8, 51.0, 35.4, 0.5],
                     [35.1, 11.5, 39.1, 15.7, 0.5], [35.6, 11.8, 39.3, 14.2, 0.5], [35.3, 11.5, 39.9, 14.5, 0.4],
                     [35.2, 11.7, 39.7, 15.7, 0.3]], dtype=np.float32)  # nms.py:24-34
    keep = R['nms_ext'].nms(torch.from_numpy(dets), 0.6).numpy()
    assert len(keep) == 3
    rng = np.random.RandomState(7)
    rnd = np.concatenate([rng.uniform(0, 200, (400, 2)), rng.uniform(5, 60, (400, 2)), rng.uniform(0.05, 1, (400, 1))], 1).astype(np.float32)
    rnd[:, 2:4] += rnd[:, 0:2]
    keep_rnd = R['nms_ext'].nms(torch.from_numpy(rnd), 0.3).numpy()
    from lfd.model.losses.iou_loss import bbox_overlaps
    b1 = torch.FloatTensor([[0, 0, 10, 10], [10, 10, 20, 20], [32, 32, 38, 42]])
    b2 = torch.FloatTensor([[0, 0, 10, 20], [0, 10, 10, 19], [10, 10, 20, 20]])
    torch.save(dict(nms_doc_dets=dets, nms_doc_keep=keep, nms_rand_dets=rnd, nms_rand_keep=keep_rnd, nms_rand_thr=0.3,
                    overlaps_b1=b1, overlaps_b2=b2, overlaps=bbox_overlaps(b1, b2)), os.path.join(out_dir, 'known_answers.pt'))
    print('known answers: doc keep', keep.tolist(), 'random keep', len(keep_rnd))
    reference_nms_case(R['nms_ext'], out_dir)

    for name, (n, h, w, cls_bias) in FORWARD_CASES.items():
        forward_case(R, name, n, h, w, cls_bias, out_dir)

    for name, (h, w) in ASSIGN_CASES.items():
        cfg = orc.CONFIGS[name]
        model = build_ref_model(R, cfg)
        sizes = sizes_for(cfg, h, w)
        pts = model.generate_point_coordinates(dict(enumerate(sizes)))
        ann = synth.synth_annotations(3, h, w, cfg['lfd']['num_classes'], seed=5, max_boxes=30)
        ct, rt = model.annotation_to_target(pts, [torch.from_numpy(a[0]) for a in ann], [torch.from_numpy(a[1]) for a in ann])
        imgs = []
        for i in range(ct.shape[0]):
            nz = torch.nonzero(ct[i].abs().sum(-1) > 0).squeeze(1)
            pos = torch.nonzero((ct[i].min(-1)[0] >= 0) & (ct[i].max(-1)[0] >= 0.001)).squeeze(1)
            imgs.append(dict(nz_rows=nz, nz_cls=ct[i][nz].clone(), pos_rows=pos, pos_reg=rt[i][pos].clone()))
        torch.save(dict(cfg=name, H=h, W=w, sizes=sizes, ann=ann, images=imgs),
                   os.path.join(out_dir, 'assign_%s.pt' % name))
        print('assign %s: P=%d pos=%s nz=%s' % (name, ct.shape[1], [int(im['pos_rows'].numel()) for im in imgs],
                                                 [int(im['nz_rows'].numel()) for im in imgs]))


if __name__ == '__main__':
    main()
