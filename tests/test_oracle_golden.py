"""CPU: the oracle restatement (oracle/*.py) against golden vectors produced by executing the reference's own
Python (tests/golden/make_golden.py).  No GPU, no /root/reference needed."""
import numpy as np
import pytest
from conftest import golden, golden_rel_err, checksum, rel_err
from oracle import relation_np as R, learn_nms_np as L, proposal_np as P

REL_CASES = ['relation_cfg0_ref', 'relation_cfg0_fanin', 'relation_n300_d1024', 'relation_n120_m100']


def _rel_case(g):
    M = int(g['M']); N = int(g['N'])
    c = R.make_relation_case(int(g['seed']), N, int(g['d']), int(g['H']), init=str(g['init']),
                             M=None if M == N else M)
    assert abs(checksum(c) - float(g['input_checksum'])) < 1e-6 * abs(float(g['input_checksum'])), 'generator drift'
    return c, N, M


@pytest.mark.parametrize('name', REL_CASES)
def test_relation_oracle_matches_reference_execution(name):
    g = golden(name)
    c, N, M = _rel_case(g)
    H = int(g['H'])
    eps = R.position_matrix(c['boxes'], M)
    np.testing.assert_allclose(eps[:g['position_matrix'].shape[0]], g['position_matrix'], rtol=1e-5, atol=1e-5)
    phi = R.position_embedding(eps[:g['position_embedding'].shape[0]])
    np.testing.assert_allclose(phi, g['position_embedding'], rtol=0, atol=2e-4)   # sin/cos of args up to +-690 in fp32
    args = (c['X'], c['boxes'], c['Wq'], c['bq'], c['Wk'], c['bk'], c['Wg'], c['bg'], c['Wout'], c['bout'])
    att = R.relation_forward(*args, key_index=M, group=H)
    assert golden_rel_err(att, g, 'attention') < 2e-5
    out = R.relation_forward(*args, key_index=M, group=H, residual_relu=True)
    assert golden_rel_err(out, g, 'out') < 2e-5
    # fp64 twin and the reordered (V' = V.Wout^T, g*exp(s)) form the CUDA kernel evaluates agree to rounding
    att64 = R.relation_forward(*args, key_index=M, group=H, dtype=np.float64)
    re64 = R.relation_forward_reordered(*args, key_index=M, group=H, dtype=np.float64)
    assert rel_err(re64, att64) < 1e-10
    # float32 reference arithmetic is itself ~3e-4 (max-norm) away from exact: sin/cos of 100*eps up to +-690 rad
    # lose ~5e-5 rad to argument rounding and log(max(relu(x),1e-6)) amplifies it for barely-alive geometry units
    assert rel_err(att, att64) < 1e-3


def test_relation_self_consistency():
    c = R.make_relation_case(5, 64, 256, 4)
    args = (c['Wq'], c['bq'], c['Wk'], c['bk'], c['Wg'], c['bg'], c['Wout'], c['bout'])
    r = R.relation_forward(c['X'], c['boxes'], *args, group=4, return_all=True, dtype=np.float64)
    np.testing.assert_allclose(r['softmax'].sum(axis=2), 1.0, atol=1e-12)
    # translation invariance of the geometry; permutation equivariance when N == M
    sh = c['boxes'].astype(np.float64) + np.array([13.0, -7.0, 13.0, -7.0])
    np.testing.assert_allclose(R.position_matrix(sh, dtype=np.float64), R.position_matrix(c['boxes'], dtype=np.float64),
                               atol=1e-9)
    perm = np.random.default_rng(0).permutation(64)
    o1 = R.relation_forward(c['X'], c['boxes'], *args, group=4, dtype=np.float64)
    o2 = R.relation_forward(c['X'][perm], c['boxes'][perm], *args, group=4, dtype=np.float64)
    np.testing.assert_allclose(o2, o1[perm], atol=1e-10)
    # identical boxes -> eps = (log 1e-3, log 1e-3, 0, 0)
    same = np.tile(c['boxes'][:1], (3, 1))
    e = R.position_matrix(same, dtype=np.float64)
    np.testing.assert_allclose(e[0, 1], [np.log(1e-3), np.log(1e-3), 0, 0], atol=1e-12)


@pytest.mark.parametrize('name', ['learn_nms_r300_c80', 'learn_nms_r60_c8'])
def test_learn_nms_oracle_matches_reference_execution(name):
    g = golden(name)
    c = L.make_learn_nms_case(int(g['seed']), R=int(g['R']), C=int(g['C']), init=str(g['init']))
    assert abs(checksum(dict(c, **c['P'])) - float(g['input_checksum'])) < 1e-6 * float(g['input_checksum'])
    multi, sbbox, sscore, final = L.learn_nms_forward(
        c['cls_score'], c['bbox_pred'], c['rois'], c['im_info'], c['feat'], c['P'], first_n=int(g['first_n']),
        num_fg_classes=int(g['C']), nongt_dim=int(g['R']))
    np.testing.assert_allclose(sscore, g['sorted_score'], rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(sbbox, g['sorted_bbox'], rtol=1e-5, atol=1e-3)
    assert rel_err(multi, g['nms_multi_score']) < 5e-5
    assert rel_err(final, g['final_score']) < 5e-5
    # pruned classes are exactly zero in both
    assert np.array_equal(multi.max(axis=(0, 2)) > 0, g['nms_multi_score'].max(axis=(0, 2)) > 0)


@pytest.mark.parametrize('name', ['proposal_38x63', 'proposal_small'])
def test_proposal_oracle_matches_reference_execution(name):
    g = golden(name)
    scales = tuple(int(s) for s in g['scales'])
    cls_prob, bbox_pred, info = P.make_proposal_case(int(g['seed']), H=int(g['H']), W=int(g['W']), A=3 * len(scales),
                                                     im_info=tuple(g['im_info'][0]))
    assert abs(checksum(dict(a=cls_prob, b=bbox_pred)) - float(g['input_checksum'])) < 1e-6 * float(g['input_checksum'])
    np.testing.assert_array_equal(P.generate_anchors(16, (0.5, 1, 2), scales), g['anchors'])
    rois, sc, aux = P.proposal_forward(cls_prob, bbox_pred, info, scales=scales, pre_nms_top_n=int(g['pre']),
                                       post_nms_top_n=int(g['post']), return_aux=True)
    # scores identify the selected anchors exactly (scores are unique): bit-exact proposal indices
    k = aux['n_kept']
    np.testing.assert_array_equal(sc[:k], g['scores'][:k])
    # coordinates: the reference's float32 np.exp may differ from the correctly-rounded one by 1 ulp
    np.testing.assert_allclose(rois[:k], g['rois'][:k], rtol=2e-6, atol=1e-4)


def test_proposal_target_oracle_matches_reference_execution():
    g = golden('proposal_target_300_7')
    rois, label, bt, bw = P.proposal_target_forward(g['rois'], g['gt_boxes'])
    np.testing.assert_array_equal(rois, g['rois_out'])
    np.testing.assert_array_equal(label, g['label'])
    np.testing.assert_array_equal(bw, g['bbox_weight'])
    np.testing.assert_allclose(bt, g['bbox_target'], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(P.bbox_overlaps(g['rois'][:, 1:], g['gt_boxes'][:, :4]), g['overlaps_py'], rtol=1e-14)


def test_misc_helpers_match_reference_execution():
    g = golden('misc_helpers')
    np.testing.assert_allclose(L.refine_boxes(g['boxes'], g['deltas'], g['im_info'])[:, :, 0], g['refined'][:, :, 0],
                               rtol=1e-6, atol=1e-4)
    np.testing.assert_allclose(L.refine_boxes(g['boxes'], g['deltas'], g['im_info'], (0, 0, 0, 0), (.1, .1, .2, .2)),
                               g['refined_ms'], rtol=1e-6, atol=1e-4)
    np.testing.assert_allclose(L.rank_embedding(100), g['rank_embedding'], atol=1e-5)
    sb = g['sorted_bbox']
    for c in range(sb.shape[1]):
        np.testing.assert_allclose(R.position_matrix(sb[:, c]), g['multi_position_matrix'][c], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(P.decode_boxes(g['boxes'].astype(np.float64), g['deltas']), g['decoded'], rtol=1e-6)
    np.testing.assert_allclose(P.encode_boxes(g['boxes'], g['boxes'][::-1].copy()), g['encoded'], rtol=1e-6, atol=1e-6)


def test_nms_multi_target_oracle_matches_reference_execution():
    g = golden('nms_multi_target')
    out = L.nms_multi_target(g['bbox'], g['gt_box'], g['score'], g['target_thresh'])
    assert out.sum() > 10
    np.testing.assert_array_equal(out, g['target'])
    # a class without gt boxes, and a gt nobody overlaps, produce no positives
    gt2 = g['gt_box'].copy(); gt2[0, :, :4] += 5000
    assert L.nms_multi_target(g['bbox'], gt2, g['score'], g['target_thresh']).sum() == 0


def test_torch_oracle_forward_equals_numpy_oracle():
    """oracle/relation_torch.py (autograd oracle of rn_relation_bwd) restates the same function as relation_np."""
    import torch
    from oracle import relation_np as R, relation_torch as RT
    for seed, N, d, H, M, res in ((3, 70, 256, 4, 50, True), (4, 60, 128, 16, None, False)):
        c = R.make_relation_case(seed, N, d, H, M=M)
        args = [c[k] for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]
        ref = R.relation_forward(*args, key_index=M, group=H, residual_relu=res, dtype=np.float64)
        out = RT.relation_forward(*[torch.tensor(a, dtype=torch.float64) for a in args], key_index=M, group=H, residual_relu=res)
        assert np.abs(out.numpy() - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())


def _deform_conv_case(seed, B=2, C=8, H=9, W=11, Co=6, dg=2, scale=0.6):
    rng = np.random.RandomState(seed)
    data = rng.randn(B, C, H, W).astype(np.float32)
    offset = (rng.randn(B, dg * 18, H, W) * scale).astype(np.float32)
    weight = (rng.randn(Co, C, 3, 3) * 0.2).astype(np.float32)
    dout = rng.randn(B, Co, H, W).astype(np.float32)
    return data, offset, weight, dout


def test_oracle_deform_conv_backward_equals_autograd():
    """C restatement of the reference's col2im / col2im_coord kernels == autograd through the (C-oracle-checked) forward."""
    import torch
    from oracle import rois_np as RO, rois_torch as RT
    data, offset, weight, dout = _deform_conv_case(5)
    t = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (data, offset, weight)]
    out = RT.deform_conv(t[0], t[1], t[2], num_deformable_group=2)
    fwd = RO.deform_conv(data, offset, weight, num_deformable_group=2)
    assert np.abs(out.detach().numpy() - fwd).max() <= 1e-4
    out.backward(torch.tensor(dout, dtype=torch.float64))
    dd, do, dw = RO.deform_conv_backward(dout, data, offset, weight, num_deformable_group=2, weight_grad_deformed=True)
    for got, want, name in ((dd, t[0].grad, 'data'), (do, t[1].grad, 'offset'), (dw, t[2].grad, 'weight')):
        assert rel_err(got, want.numpy()) <= 1e-4, name
    # the reference's dWeight (deformable_convolution-inl.h:215) is the gradient of the UN-deformed dilated convolution
    tw = torch.tensor(weight, dtype=torch.float64, requires_grad=True)
    torch.nn.functional.conv2d(torch.tensor(data, dtype=torch.float64), tw, padding=2, dilation=2).backward(
        torch.tensor(dout, dtype=torch.float64))
    dw_ref = RO.deform_conv_backward(dout, data, offset, weight, num_deformable_group=2)[2]
    assert rel_err(dw_ref, tw.grad.numpy()) <= 1e-4


def test_oracle_deform_psroi_backward_equals_autograd():
    import torch
    from oracle import rois_np as RO, rois_torch as RT
    rng = np.random.RandomState(9)
    B, C, H, W, R, P = 2, 8, 12, 16, 10, 3
    data = rng.randn(B, C, H, W).astype(np.float32)
    x1 = rng.uniform(0, 150, R); y1 = rng.uniform(0, 100, R)
    rois = np.stack([rng.randint(0, B, R), x1, y1, x1 + rng.uniform(20, 100, R), y1 + rng.uniform(20, 90, R)], 1).astype(np.float32)
    trans = rng.randn(R, 2, P, P).astype(np.float32)
    kw = dict(spatial_scale=0.0625, output_dim=C, group_size=1, pooled_size=P, sample_per_part=2, trans_std=0.1)
    for tr in (None, trans):
        out, cnt = RO.deform_psroi_pool(data, rois, tr, **kw)
        dout = rng.randn(*out.shape).astype(np.float32)
        td = torch.tensor(data, dtype=torch.float64, requires_grad=True)
        tt = None if tr is None else torch.tensor(tr, dtype=torch.float64, requires_grad=True)
        o, c = RT.deform_psroi_pool(td, torch.tensor(rois, dtype=torch.float64), tt, **kw)
        assert np.abs(o.detach().numpy() - out).max() <= 1e-5 and np.array_equal(c.numpy(), cnt)
        o.backward(torch.tensor(dout, dtype=torch.float64))
        dd, dt = RO.deform_psroi_pool_backward(dout, cnt, data, rois, tr, **kw)
        assert rel_err(dd, td.grad.numpy()) <= 1e-5
        if tr is not None:
            assert rel_err(dt, tt.grad.numpy()) <= 1e-4


def test_oracle_roi_pool_backward_routes_to_argmax():
    import torch
    from oracle import rois_np as RO
    rng = np.random.RandomState(2)
    data = rng.randn(2, 4, 20, 30).astype(np.float32)
    rois = np.array([[0, 10, 20, 300, 200], [1, 100, 50, 400, 310], [0, 0, 0, 479, 319]], np.float32)
    out, arg = RO.roi_pool(data, rois, (7, 7), 0.0625)
    dout = rng.randn(*out.shape).astype(np.float32)
    dd = RO.roi_pool_backward(dout, arg, rois, data.shape)
    # max pooling: d out / d data is 1 at the argmax; compare with a direct scatter in float64
    want = np.zeros(data.shape, np.float64)
    for n in range(3):
        for c in range(4):
            for p in range(49):
                a = arg[n, c].reshape(-1)[p]
                if a >= 0:
                    want[int(rois[n, 0]), c].reshape(-1)[a] += dout[n, c].reshape(-1)[p]
    assert rel_err(dd, want) <= 1e-6


def test_torch_learn_nms_forward_equals_numpy_oracle():
    import torch
    from oracle import learn_nms_np as LN, learn_nms_torch as LT
    c = LN.make_learn_nms_case(7, R=60, C=8, d=256)
    c['P']['roi_feat_embedding_weight'] = c['P']['roi_feat_embedding_weight'][:, :256].copy()
    want = LN.learn_nms_forward(c['cls_score'], c['bbox_pred'], c['rois'], c['im_info'], c['feat'], c['P'], first_n=20,
                                num_fg_classes=8, class_thresh=0.0, nongt_dim=50, dtype=np.float64)
    P = {k: torch.tensor(v, dtype=torch.float64) for k, v in c['P'].items()}
    multi, ss, order = LT.learn_nms_forward(torch.tensor(c['cls_score'], dtype=torch.float64), c['bbox_pred'], c['rois'],
                                            c['im_info'], torch.tensor(c['feat'], dtype=torch.float64), P, first_n=20,
                                            num_fg_classes=8, class_thresh=0.0, nongt_dim=50)
    assert np.abs(multi.numpy() - want[0]).max() <= 1e-10
    assert np.abs(ss.numpy() - want[2]).max() <= 1e-12


def test_ohem_oracle_matches_reference_execution():
    """oracle/train_np.box_annotator_ohem == the reference's BoxAnnotatorOHEMOperator.forward run under the numpy shim"""
    from oracle import train_np as TN
    g = golden('box_annotator_ohem')
    lab, w, _ = TN.box_annotator_ohem(g['cls_score'], g['bbox_pred'], g['labels'], g['bbox_targets'], g['bbox_weights'],
                                      int(g['roi_per_img']))
    assert np.array_equal(lab, g['labels_ohem']) and np.array_equal(w, g['bbox_weights_ohem'])
    assert int((lab >= 0).sum()) == int(g['roi_per_img'])


def test_nms_loss_oracle_gradient_is_autograd():
    import torch
    from oracle import train_np as TN, learn_nms_torch as LT
    rng = np.random.default_rng(3)
    m = rng.uniform(0.0, 1.0, (30, 8, 5)).astype(np.float32); t = (rng.random((30, 8, 5)) < 0.1).astype(np.float32)
    pos, neg, d = TN.nms_loss(m, t, 30, 5, loss_scale=1.0, pos_grad_scale=4.0)
    tm = torch.tensor(m, dtype=torch.float64, requires_grad=True)
    p, n = LT.nms_loss(tm, torch.tensor(t, dtype=torch.float64), 30, 5)
    (4.0 * p.sum() + n.sum()).backward()
    assert rel_err(pos, p.detach().numpy()) <= 1e-5 and rel_err(neg, n.detach().numpy()) <= 1e-5
    assert rel_err(d, tm.grad.numpy()) <= 1e-5


def test_relation_oracle_matches_fpn_reference_execution():
    """row a4: the FPN symbol's own extract_position_matrix / attention_module_multi_head (keys = take(non_gt_index), pair FC
    as a 1x1 convolution) executed under the shim == oracle relation_forward(key_index=...)"""
    from oracle import relation_np as R
    g = golden('relation_fpn_n90_k70')
    c = R.make_relation_case(int(g['seed']), int(g['N']), int(g['d']), int(g['H']), init='fan_in')
    assert abs(checksum(c) - float(g['input_checksum'])) <= 1e-6 * abs(float(g['input_checksum']))
    args = [c[k] for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]
    out = R.relation_forward(*args, key_index=g['non_gt_index'], group=int(g['H']), residual_relu=False, dtype=np.float32)
    assert rel_err(out, g['attention']) < 2e-5
    pm = R.position_matrix(c['boxes'], key_index=g['non_gt_index'])[:8]
    assert rel_err(pm, g['position_matrix']) < 1e-6


def test_learn_nms_oracle_matches_reference_execution_non_gt_index():
    """FPN form of the op (has_non_gt_index=True, 20 inputs, train-time means/stds): LNMS:260-283"""
    g = golden('learn_nms_nongt_index')
    c = L.make_learn_nms_case(int(g['seed']), R=int(g['R']), C=int(g['C']), init='fan_in')
    multi, sbbox, sscore, _ = L.learn_nms_forward(c['cls_score'], c['bbox_pred'], c['rois'], c['im_info'], c['feat'], c['P'],
                                                  first_n=int(g['first_n']), num_fg_classes=int(g['C']), means=g['means'],
                                                  stds=g['stds'], non_gt_index=g['non_gt_index'])
    assert np.array_equal(sscore, g['sorted_score']) and np.abs(sbbox - g['sorted_bbox']).max() <= 1e-4
    assert rel_err(multi, g['nms_multi_score']) < 2e-5


def test_product_synth_generator_equals_oracle_generator():
    """bench.py / tools draw their synthetic relation cases from relnet_b200.synth (so the product never imports oracle);
    the parity tests draw theirs from oracle.relation_np: same seeds must give the same bits."""
    import relnet_b200.synth as S
    from oracle import relation_np as R
    for kw in (dict(seed=2, N=30, d=64, H=4), dict(seed=5, N=17, d=128, H=16, init='ref', dq=1024, dout=128)):
        a, b = S.make_relation_case(**kw), R.make_relation_case(**kw)
        assert a.keys() == b.keys()
        for k in a:
            assert np.array_equal(a[k], b[k]), k

