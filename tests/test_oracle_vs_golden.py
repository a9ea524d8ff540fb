# -*- coding: utf-8 -*-
"""CPU tests: the oracle restatement (oracle/lfd_oracle.py) against vectors produced by the REFERENCE's own modules
(tests/gen_golden.py) and against the reference's docstring known answers."""
import numpy as np
import pytest
import torch

import synth
from helpers import load_golden, build_model, rel_err
from oracle import lfd_oracle as orc
from oracle import build_ref

FWD = ['WIDERFACE_XS', 'WIDERFACE_S', 'WIDERFACE_L', 'TT100K_L', 'TL_L', 'TEST_FAST', 'TEST_FASTEST']


@pytest.mark.parametrize('name', FWD)
def test_state_dict_keys_match_reference(name):
    g = load_golden('forward_%s.pt' % name)
    sd = build_model(name).state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(k, tuple(s)) for k, s in g['keys']]
    syn = synth.synth_state_dict(sd, seed=g['seed'], cls_bias=g['cls_bias'])
    assert abs(synth.state_checksum(syn) - g['checksum']) <= 1e-6 * g['checksum'], 'RNG drift: regenerate goldens'


@pytest.mark.parametrize('name', FWD)
def test_forward_fp32_matches_reference(name):
    g = load_golden('forward_%s.pt' % name)
    cfg = orc.CONFIGS[name]
    sd = synth.synth_state_dict(build_model(name).state_dict(), seed=g['seed'], cls_bias=g['cls_bias'])
    x = synth.synth_input(g['N'], g['H'], g['W'])
    cls, reg, sizes = orc.forward(cfg, sd, x)
    assert [tuple(s) for s in sizes] == [tuple(s) for s in g['sizes']]
    assert rel_err(cls, g['cls'])[0] < 2e-5 and rel_err(reg, g['reg'])[0] < 2e-5


@pytest.mark.parametrize('name', FWD)
def test_bf16_emulation_drift_is_bounded(name):
    """Gate C (reported): bf16 pipeline vs the fp32 reference forward -- bounded drift, not parity."""
    g = load_golden('forward_%s.pt' % name)
    cfg = orc.CONFIGS[name]
    sd = synth.synth_state_dict(build_model(name).state_dict(), seed=g['seed'], cls_bias=g['cls_bias'])
    x = synth.synth_input(g['N'], g['H'], g['W'])
    cls, reg, _ = orc.forward(cfg, sd, x, emulate_bf16=True)
    assert rel_err(cls, g['cls'])[1] < 5e-2 and rel_err(reg, g['reg'])[1] < 5e-2


@pytest.mark.parametrize('name', FWD)
def test_results_match_reference(name):
    g = load_golden('forward_%s.pt' % name)
    cfg = orc.CONFIGS[name]
    for (thr, iou), ref in g['results'].items():
        res, _ = orc.get_results(cfg, g['cls'], g['reg'], g['sizes'], g['meta'], thr, iou)
        for i in range(g['N']):
            a, b = np.asarray(res[i], np.float64).reshape(-1, 6), ref[i].double().numpy()
            assert a.shape == b.shape, (name, thr, iou, i, a.shape, b.shape)
            if a.size:
                assert np.array_equal(a[:, 0], b[:, 0])
                np.testing.assert_allclose(a[:, 1:], b[:, 1:], rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize('name', ['WIDERFACE_S', 'WIDERFACE_L', 'TT100K_L'])
def test_label_assignment_matches_reference(name):
    g = load_golden('assign_%s.pt' % name)
    cfg = orc.CONFIGS[name]
    for (boxes, labels), im in zip(g['ann'], g['images']):
        ct, rt = orc.assign_targets(cfg, g['sizes'], boxes, labels)
        nz = np.nonzero(np.abs(ct).sum(-1) > 0)[0]
        assert np.array_equal(nz, im['nz_rows'].numpy())
        ref = im['nz_cls'].numpy()
        # structure (gray = -1, background = 0, green > 0) is exact; green score VALUES agree to 2 ulp only, because
        # torch's vectorised CPU sqrt is not correctly rounded (differs from IEEE sqrt on ~0.7 % of inputs)
        assert np.array_equal(np.sign(ct[nz]), np.sign(ref)) and np.array_equal(ct[nz] == -1, ref == -1)
        np.testing.assert_allclose(ct[nz], ref, rtol=3e-7, atol=0)
        pos = np.nonzero((ct.min(-1) >= 0) & (ct.max(-1) >= 0.001))[0]
        assert np.array_equal(pos, im['pos_rows'].numpy())
        assert np.array_equal(rt[pos], im['pos_reg'].numpy())


@pytest.mark.parametrize('name', FWD)
def test_loss_and_gradients_match_reference(name):
    g = load_golden('forward_%s.pt' % name)
    cfg = orc.CONFIGS[name]
    cls = g['cls'].clone().requires_grad_(True)
    reg = g['reg'].clone().requires_grad_(True)
    out = orc.get_loss(cfg, cls, reg, g['sizes'], g['ann'])
    out['loss'].backward()
    lv = g['loss_values']
    assert abs(float(out['loss']) - lv['loss']) <= 1e-5 * abs(lv['loss'])
    assert abs(float(out['classification_loss']) - lv['classification_loss']) <= 1e-5 * abs(lv['classification_loss'])
    assert abs(float(out['regression_loss']) - lv['regression_loss']) <= 1e-5 * max(abs(lv['regression_loss']), 1e-6)
    assert rel_err(cls.grad, g['grad_cls'])[0] < 1e-5
    assert rel_err(reg.grad, g['grad_reg'])[0] < 1e-4 or float(g['grad_reg'].abs().max()) == 0.0


def test_known_answers():
    k = load_golden('known_answers.pt')
    assert orc.nms(k['nms_doc_dets'], 0.6).tolist() == k['nms_doc_keep'].tolist() == [0, 3, 4]   # nms.py:24-34
    assert orc.nms(k['nms_rand_dets'], k['nms_rand_thr']).tolist() == k['nms_rand_keep'].tolist()
    ov = orc.bbox_overlaps(k['overlaps_b1'], k['overlaps_b2'])                                      # iou_loss.py:28-42
    assert torch.allclose(ov, k['overlaps']) and torch.allclose(ov, torch.tensor([[0.5, 0, 0], [0, 0, 1.0], [0, 0, 0]]))
    empty, nonempty = torch.zeros((0, 4)), torch.tensor([[0., 0, 10, 9]])
    assert tuple(orc.bbox_overlaps(empty, nonempty).shape) == (0, 1) and tuple(orc.bbox_overlaps(nonempty, empty).shape) == (1, 0)
    # losses/utils.py:67-85
    pred, target, weight = torch.tensor([0., 2, 3]), torch.tensor([1., 1, 1]), torch.tensor([1., 0, 1])
    l1 = (pred - target).abs()
    assert abs(float(orc.weight_reduce_loss(l1)) - 1.3333) < 1e-4
    assert float(orc.weight_reduce_loss(l1, weight)) == 1.0
    assert orc.weight_reduce_loss(l1, reduction='none').tolist() == [1., 1., 2.]
    assert float(orc.weight_reduce_loss(l1, weight, avg_factor=2)) == 1.5
    with pytest.raises(ValueError):
        orc.weight_reduce_loss(l1, weight, reduction='sum', avg_factor=2)


def test_reference_cpu_nms_binary_agrees_with_oracle():
    """The reference's own nms_cpu.cpp, through its outputs stored by tests/gen_golden.py; where oracle/_ref holds the compiled
    binary, it must still reproduce them."""
    cases = load_golden('reference_nms.pt')
    assert sorted({len(c['dets']) for c in cases}) == [1, 7, 300] and sorted({c['thr'] for c in cases}) == [0.3, 0.6]
    mod = build_ref.load_module()
    for c in cases:
        keep = c['keep'].tolist()
        assert orc.nms(c['dets'], c['thr']).tolist() == keep, (len(c['dets']), c['thr'])
        if mod is not None:
            assert mod.nms(torch.from_numpy(c['dets']), c['thr']).tolist() == keep


def test_focal_restatement_pinned_against_torchvision():
    """The reference has no CPU focal loss; the restatement of the .cu is pinned against torchvision's independent one."""
    from torchvision.ops import sigmoid_focal_loss as tv_focal
    g = torch.Generator().manual_seed(1)
    for C in (1, 45):
        x = (torch.randn((200, C), generator=g) * 4).requires_grad_(True)
        t = torch.randint(0, C + 1, (200,), generator=g)
        onehot = torch.zeros((200, C + 1)).scatter_(1, t[:, None], 1.0)[:, :C]
        ref = tv_focal(x, onehot, alpha=0.25, gamma=2.0, reduction='none')
        mine = orc.sigmoid_focal_loss_forward(x.detach(), t, 2.0, 0.25)
        assert float((ref - mine).abs().max()) < 5e-6
        (ref.sum()).backward()
        gb = orc.sigmoid_focal_loss_backward(x.detach(), t, torch.ones_like(mine), 2.0, 0.25)
        assert float((x.grad - gb).abs().max()) < 5e-6
