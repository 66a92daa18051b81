"""GPU: the CUDA path (through the C ABI) against the CPU oracle and the committed golden vectors.

Tolerances (also in DESIGN.md):
  * indices / labels / kept sets / pruned-class masks: bit-exact
  * relation-module float outputs: max|a-b| / max|b| <= 1e-3 against the FLOAT32 oracle / golden, i.e. the reference's
    own arithmetic (north_star: "within 1e-3 rel on relation-module fp32 outputs for identical inputs"); the fp32 parity
    mode is held to 3e-4.  The float64 twin is reported but not the target: float32 evaluation of the geometry is
    ill-conditioned for near-concentric boxes (cx_n - cx_m cancels, x100 inside sin/cos), so the reference itself
    sits up to ~5e-3 away from exact arithmetic on these inputs (measured on the oracle, see DESIGN.md).
  * ROI / deformable kernels (compiled without FMA, same op order as the C oracle): 1e-5 relative
"""
import numpy as np
import pytest
import torch
from conftest import golden, golden_rel_err, rel_err
from oracle import relation_np as R, learn_nms_np as L, proposal_np as P, rois_np as RO

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops(cuda_device):
    import __graft_entry__ as g
    g.build()
    import relnet_b200
    torch.cuda.set_device(cuda_device)
    return relnet_b200.ops


def precisions(ops):
    import os
    if os.environ.get('RELNET_TEST_PREC'):
        return os.environ['RELNET_TEST_PREC'].split(',')
    return ['fp32', 'f16'] if ops.device_info()['sm100'] else ['fp32']


def T(a, dev='cuda'):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def rel_args(c):
    return [c[k] for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]


# ------------------------------------------------------------------------------------------------ tcgen05 plumbing
def test_umma_selftest(ops):
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 needs sm_100')
    rng = np.random.default_rng(0)
    a = rng.standard_normal((128, 64)).astype(np.float16); b = rng.standard_normal((128, 64)).astype(np.float16)
    p = rng.random((128, 128)).astype(np.float16); v = rng.standard_normal((128, 64)).astype(np.float16)
    s, o = ops.umma_selftest(T(a), T(b), T(p), T(v))
    torch.cuda.synchronize()
    s_ref = a.astype(np.float64) @ b.astype(np.float64).T
    o_ref = p.astype(np.float64) @ v.astype(np.float64)
    assert rel_err(s.cpu().numpy(), s_ref) < 1e-5, 'K-major SW128 UMMA / TMA / TMEM mapping is wrong'
    assert rel_err(o.cpu().numpy(), o_ref) < 1e-5, 'MN-major B / manually swizzled A is wrong'


# ------------------------------------------------------------------------------------------------ geometry
def test_pos_embed_matches_oracle(ops):
    rng = np.random.default_rng(3)
    boxes = R.make_boxes(rng, 77)
    eps, emb = ops.pos_embed(T(boxes), M=60)
    e_ref = R.position_matrix(boxes, 60, dtype=np.float32)
    np.testing.assert_allclose(eps.cpu().numpy(), e_ref, rtol=2e-6, atol=2e-6)
    phi_ref = R.position_embedding(eps.cpu().numpy(), dtype=np.float64)   # same eps -> isolates the sin/cos evaluation
    np.testing.assert_allclose(emb.cpu().numpy(), phi_ref, atol=1e-4)     # args up to 690 rad: 1 ulp of the argument
    same = np.tile(boxes[:1], (3, 1))
    eps, _ = ops.pos_embed(T(same), want_emb=False)
    np.testing.assert_allclose(eps.cpu().numpy()[0, 1], [np.log(1e-3), np.log(1e-3), 0, 0], atol=1e-6)


@pytest.mark.parametrize('H', [4, 16])
def test_geometry_weight_matches_oracle(ops, H):
    c = R.make_relation_case(9, 150, 64 * H, H)
    g = ops.geometry_weight(T(c['boxes']), T(c['Wg']), T(c['bg']), M=120)
    ref = R.geometry_weight(c['boxes'], c['Wg'], c['bg'], 120, dtype=np.float32).transpose(1, 0, 2)    # [H,N,M]
    np.testing.assert_allclose(g.cpu().numpy(), ref, rtol=1e-3, atol=1e-4)
    assert rel_err(g.cpu().numpy(), ref) < 1e-4


# ------------------------------------------------------------------------------------------------ relation module
REL_GOLDEN = ['relation_cfg0_ref', 'relation_cfg0_fanin', 'relation_n300_d1024', 'relation_n120_m100']


@pytest.mark.parametrize('name', REL_GOLDEN)
def test_relation_matches_golden_and_oracle(ops, name):
    g = golden(name)
    N, M, H = int(g['N']), int(g['M']), int(g['H'])
    c = R.make_relation_case(int(g['seed']), N, int(g['d']), H, init=str(g['init']), M=None if M == N else M)
    args = rel_args(c)
    ref64 = R.relation_forward(*args, key_index=M, group=H, dtype=np.float64)
    print('%s: float32 reference arithmetic vs float64: %.2e' % (name, golden_rel_err(ref64, g, 'attention')))
    # a fixture with a subset of rows: every row is held to the float32 oracle, which test_oracle_golden ties to those rows
    ref32 = R.relation_forward(*args, key_index=M, group=H) if 'rows' in g else None
    for prec in precisions(ops):
        att = ops.relation(*[T(a) for a in args], M=M, group=H, precision=prec).cpu().numpy()
        out = ops.relation(*[T(a) for a in args], M=M, group=H, residual_relu=True, precision=prec).cpu().numpy()
        e_gold, e64 = golden_rel_err(att, g, 'attention'), rel_err(att, ref64)
        print('%s[%s]: attention rel err vs golden(fp32 ref exec) %.2e, vs fp64 oracle %.2e' % (name, prec, e_gold, e64))
        assert e_gold < 1e-3
        assert golden_rel_err(out, g, 'out') < 1e-3
        if ref32 is not None:
            assert rel_err(att, ref32) < 1e-3 and rel_err(out, np.maximum(c['X'] + ref32, 0)) < 1e-3
        if prec == 'fp32':
            assert e_gold < 3e-4
            assert ref32 is None or rel_err(att, ref32) < 3e-4


def test_relation_key_index_and_softmax(ops):
    c = R.make_relation_case(21, 90, 256, 4)
    idx = np.random.default_rng(1).permutation(90)[:50].astype(np.int32)
    args = rel_args(c)
    ref = R.relation_forward(*args, key_index=idx, group=4, dtype=np.float32, return_all=True)
    for prec in precisions(ops):
        if prec == 'f16':          # the tcgen05 path never materialises the softmax: asking for it must be loud
            with pytest.raises(Exception):
                ops.relation(*[T(a) for a in args], key_index=T(idx), group=4, precision=prec, return_softmax=True)
            out, sm = ops.relation(*[T(a) for a in args], key_index=T(idx), group=4, precision=prec), None
        else:
            out, sm = ops.relation(*[T(a) for a in args], key_index=T(idx), group=4, precision=prec, return_softmax=True)
        assert rel_err(out.cpu().numpy(), ref['attn']) < 1e-3
        if sm is not None and prec == 'fp32':
            np.testing.assert_allclose(sm.cpu().numpy().sum(-1), 1.0, atol=1e-5)
            assert rel_err(sm.cpu().numpy(), ref['softmax']) < 1e-3


def test_relation_batched_learn_nms_shape(ops):
    """batch of independent problems with d=128, dq=1024, dout=128 (the learn-NMS relation, LNMS:45-127)."""
    B, n = 5, 37
    outs, Xs, bs = [], [], []
    c0 = R.make_relation_case(40, n, 128, 16, dq=1024, dout=128)
    rng = np.random.default_rng(5)
    for b in range(B):
        X = (rng.standard_normal((n, 128)) * 0.5).astype(np.float32); bx = R.make_boxes(rng, n)
        Xs.append(X); bs.append(bx)
        a = [X, bx] + rel_args(c0)[2:]
        outs.append(R.relation_forward(*a, group=16, residual_relu=True, dtype=np.float32))
    for prec in precisions(ops):
        out = ops.relation(T(np.stack(Xs)), T(np.stack(bs)), *[T(a) for a in rel_args(c0)[2:]], group=16,
                           residual_relu=True, precision=prec).cpu().numpy()
        assert rel_err(out, np.stack(outs)) < 1e-3


@pytest.mark.parametrize('N,d,H', [(1000, 256, 4), (300, 256, 16), (515, 1024, 16)])
def test_relation_sweep_points(ops, N, d, H):
    """BASELINE.json configs[4] shapes the float64 oracle finishes in seconds (odd N exercises partial tiles)."""
    c = R.make_relation_case(N * 7 + d + H, N, d, H)
    args = rel_args(c)
    ref = R.relation_forward(*args, group=H, dtype=np.float32)
    for prec in precisions(ops):
        out = ops.relation(*[T(a) for a in args], group=H, precision=prec).cpu().numpy()
        print('sweep N=%d d=%d H=%d [%s]: rel err vs float32 oracle %.2e' % (N, d, H, prec, rel_err(out, ref)))
        assert rel_err(out, ref) < 1e-3


@pytest.mark.parametrize('N,M,d,H,kidx', [(70, 50, 256, 4, False), (300, 300, 1024, 16, False), (131, 97, 256, 16, True),
                                          (300, 300, 1024, 4, False)])
def test_relation_tf32_forward_matches_oracle(ops, N, M, d, H, kidx):
    """RN_PREC_TF32: the general (materialising) kernels with every GEMM on the library's tcgen05 tf32 engine -- the forward
    that rn_relation_bwd recomputes.  Output and softmax against the float32 oracle at the relation tolerance 1e-3."""
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 needs sm_100')
    c = R.make_relation_case(N * 11 + d + H, N, d, H, M=None if (M == N or kidx) else M)
    args = rel_args(c)
    key_index = np.random.RandomState(N).permutation(N)[:M].astype(np.int32) if kidx else None
    allr = R.relation_forward(*args, key_index=key_index if kidx else M, group=H, residual_relu=True, dtype=np.float32,
                              return_all=True)
    ref, ref_sm = allr['out'], allr['softmax']
    out, sm = ops.relation(*[T(a) for a in args], key_index=T(key_index) if kidx else None, M=None if kidx else M, group=H,
                           residual_relu=True, precision='tf32', return_softmax=True)
    e, es = rel_err(out.cpu().numpy(), ref), rel_err(sm.cpu().numpy(), ref_sm)
    print('tf32 forward N=%d M=%d d=%d H=%d: out %.2e softmax %.2e' % (N, M, d, H, e, es))
    assert e < 1e-3 and es < 2e-3


def test_relation_full_size_properties(ops):
    """N=3000, d=1024 (largest sweep point): oracle-free properties -- permutation equivariance and convexity of the
    aggregation (with Wout = I, bout = 0 every output row is a convex combination of the key rows)."""
    N, d, H = 3000, 1024, 16
    c = R.make_relation_case(123, N, d, H)
    t = [T(a) for a in rel_args(c)]
    perm = torch.randperm(N, device='cuda')
    for prec in precisions(ops):
        o1 = ops.relation(*t, group=H, precision=prec)
        o2 = ops.relation(t[0][perm], t[1][perm], *t[2:], group=H, precision=prec)
        assert float((o2 - o1[perm]).abs().max() / o1.abs().max()) < 2e-3
        eye = torch.eye(d, device='cuda'); zero = torch.zeros(d, device='cuda')
        o3 = ops.relation(t[0], t[1], *t[2:8], eye, zero, group=H, precision=prec)
        lo, hi = t[0].min(0).values, t[0].max(0).values
        assert bool(((o3 >= lo - 2e-2) & (o3 <= hi + 2e-2)).all())


def test_linear_matches_numpy(ops):
    rng = np.random.default_rng(2)
    x = rng.standard_normal((300, 1024)).astype(np.float32); W = (rng.standard_normal((1024, 1024)) / 32).astype(np.float32)
    b = rng.standard_normal(1024).astype(np.float32)
    ref = np.maximum(x.astype(np.float64) @ W.astype(np.float64).T + b, 0)
    for prec in precisions(ops):
        y = ops.linear(T(x), T(W), T(b), relu=True, precision=prec).cpu().numpy()
        assert rel_err(y, ref) < (1e-5 if prec == 'fp32' else 1e-3)


# ------------------------------------------------------------------------------------------------ learn-NMS head
@pytest.mark.parametrize('name', ['learn_nms_r300_c80', 'learn_nms_r60_c8'])
def test_learn_nms_matches_golden(ops, name):
    g = golden(name)
    c = L.make_learn_nms_case(int(g['seed']), R=int(g['R']), C=int(g['C']), init=str(g['init']))
    w = {k: T(v) for k, v in c['P'].items()}
    # 'tf32' = RN_PREC_TF32: the general kernels with every GEMM on the tcgen05 tf32 engine (the forward of the training graph,
    # and the one rn_learn_nms_bwd recomputes)
    for prec in precisions(ops) + (['tf32'] if ops.device_info()['sm100'] else []):
        multi, sbbox, sscore, final = ops.learn_nms(T(c['cls_score']), T(c['bbox_pred']), T(c['rois']), T(c['im_info']),
                                                   T(c['feat']), w, first_n=int(g['first_n']), nongt_dim=int(g['R']),
                                                   precision=prec)
        np.testing.assert_allclose(sscore.cpu().numpy(), g['sorted_score'], rtol=2e-5, atol=1e-8)
        np.testing.assert_allclose(sbbox.cpu().numpy(), g['sorted_bbox'], rtol=1e-5, atol=2e-3)
        m = multi.cpu().numpy()
        assert np.array_equal(m.max(axis=(0, 2)) > 0, g['nms_multi_score'].max(axis=(0, 2)) > 0), 'class pruning differs'
        # tf32: operands truncated to 10-bit mantissas in all six GEMMs of the head.  The relation module alone measures 2e-4..1.6e-3
        # in this mode (test_relation_tf32_forward_matches_oracle); the bound for the three-stage head is a sanity bound, not yet
        # tightened against a measured value (printed below) -- the 1e-3 parity claim of the path is the fp32 / f16 rows.
        tol = 2e-2 if prec == 'tf32' else 1e-3
        print('learn_nms %s [%s]: multi %.2e final %.2e' % (name, prec, rel_err(m, g['nms_multi_score']), rel_err(final.cpu().numpy(), g['final_score'])))
        assert rel_err(m, g['nms_multi_score']) < tol
        assert rel_err(final.cpu().numpy(), g['final_score']) < tol


# ------------------------------------------------------------------------------------------------ proposal / NMS
@pytest.mark.parametrize('name', ['proposal_38x63', 'proposal_small'])
def test_proposal_matches_golden_bit_exact_indices(ops, name):
    g = golden(name)
    scales = tuple(int(s) for s in g['scales'])
    cls_prob, bbox_pred, info = P.make_proposal_case(int(g['seed']), H=int(g['H']), W=int(g['W']), A=3 * len(scales),
                                                     im_info=tuple(g['im_info'][0]))
    rois, scores, nk = ops.proposal(T(cls_prob), T(bbox_pred), T(info), scales=scales, pre_nms_top_n=int(g['pre']),
                                    post_nms_top_n=int(g['post']), return_num_kept=True)
    o_rois, o_sc, aux = P.proposal_forward(cls_prob, bbox_pred, info, scales=scales, pre_nms_top_n=int(g['pre']),
                                           post_nms_top_n=int(g['post']), return_aux=True)
    assert int(nk.item()) == aux['n_kept']
    # against the oracle: everything bit-exact (same decode definition, same tie and padding rules)
    np.testing.assert_array_equal(scores.cpu().numpy(), o_sc)
    np.testing.assert_array_equal(rois.cpu().numpy(), o_rois)
    # against the reference execution: the unique scores identify the chosen anchors -> indices bit-exact
    k = aux['n_kept']
    np.testing.assert_array_equal(scores.cpu().numpy()[:k], g['scores'][:k])
    np.testing.assert_allclose(rois.cpu().numpy()[:k], g['rois'][:k], rtol=2e-6, atol=1e-4)


def test_proposal_heavy_overlap_and_ties(ops):
    """few distinct score values (ties everywhere) + tiny deltas (heavy overlap, long NMS sweep)."""
    rng = np.random.default_rng(8)
    H, W, A = 20, 30, 12
    fg = (rng.integers(0, 16, (1, A, H, W)) / 16.0).astype(np.float32)
    cls_prob = np.concatenate([1 - fg, fg], 1)
    bbox_pred = (rng.standard_normal((1, 4 * A, H, W)) * 0.02).astype(np.float32)
    info = np.array([[320.0, 480.0, 1.0]], np.float32)
    rois, scores = ops.proposal(T(cls_prob), T(bbox_pred), T(info), pre_nms_top_n=3000, post_nms_top_n=200)
    o_rois, o_sc = P.proposal_forward(cls_prob, bbox_pred, info, pre_nms_top_n=3000, post_nms_top_n=200)
    np.testing.assert_array_equal(rois.cpu().numpy(), o_rois)
    np.testing.assert_array_equal(scores.cpu().numpy(), o_sc)


def _nms_case():
    rng = np.random.default_rng(4)
    boxes = R.make_boxes(rng, 3000)
    boxes[1000:2000] = boxes[:1000] + rng.normal(0, 3, (1000, 4)).astype(np.float32)      # near duplicates
    sc = rng.permutation(3000).astype(np.float32) / 3000
    order = np.argsort(-sc, kind='stable')
    return np.hstack([boxes, sc[:, None]])[order].astype(np.float32)


def test_nms_matches_oracle_and_reference_kernel(ops):
    dets = _nms_case()
    keep, num = ops.nms(T(dets), 0.7)
    k = keep.cpu().numpy()[:int(num.item())]
    np.testing.assert_array_equal(k, RO.nms_sorted(dets, 0.7))
    # what the REFERENCE's own lib/nms/nms_kernel.cu keeps of these boxes on a B200 (tests/golden/make_reference_kernels.py)
    g = golden('reference_gpu_nms')
    assert float(g['thresh']) == np.float32(0.7)
    np.testing.assert_array_equal(k, g['keep'])
    # early exit at max_keep: the list must be the prefix of the full sweep's list
    for mk in (50, 300, 2000):
        keep2, num2 = ops.nms(T(dets), 0.7, max_keep=mk)
        assert int(num2.item()) == min(mk, len(k))
        np.testing.assert_array_equal(keep2.cpu().numpy()[:int(num2.item())], k[:mk])
    # edge cases: single box, all identical boxes
    keep3, num3 = ops.nms(T(dets[:1]), 0.7)
    assert int(num3.item()) == 1
    same = np.tile(dets[:1], (130, 1))
    keep4, num4 = ops.nms(T(same), 0.7)
    assert int(num4.item()) == 1 and int(keep4[0].item()) == 0
    # n > 8192 with max_keep = n takes the bitmask + sweep form (lib/nms/nms_kernel.cu layout) instead of the greedy CTA
    big = np.vstack([dets, dets + np.float32(0.25), dets + np.float32(500.0)])[:9000]
    big = big[np.argsort(-big[:, 4], kind='stable')].astype(np.float32)
    keep5, num5 = ops.nms(T(big), 0.7)
    np.testing.assert_array_equal(keep5.cpu().numpy()[:int(num5.item())], RO.nms_sorted(big, 0.7))


def test_bbox_overlaps_and_proposal_target(ops):
    g = golden('proposal_target_300_7')
    ov = ops.bbox_overlaps(T(g['rois'][:, 1:]), T(g['gt_boxes'][:, :4])).cpu().numpy()
    np.testing.assert_allclose(ov, g['overlaps_py'], rtol=1e-14, atol=0)
    ro, lab, bt, bw = ops.proposal_target(T(g['rois']), T(g['gt_boxes']))
    np.testing.assert_array_equal(ro.cpu().numpy(), g['rois_out'])
    np.testing.assert_array_equal(lab.cpu().numpy(), g['label'])
    np.testing.assert_array_equal(bw.cpu().numpy(), g['bbox_weight'])
    np.testing.assert_allclose(bt.cpu().numpy(), g['bbox_target'], rtol=2e-6, atol=2e-6)


# ------------------------------------------------------------------------------------------------ ROI ops / deformable
def _roi_case(seed, nroi=300, C=64, H=38, W=63):
    rng = np.random.default_rng(seed)
    data = rng.standard_normal((1, C, H, W)).astype(np.float32)
    boxes = R.make_boxes(rng, nroi)
    rois = np.hstack([np.zeros((nroi, 1), np.float32), boxes]).astype(np.float32)
    rois[:4, 1:] = [[0, 0, 0, 0], [990, 590, 999, 599], [-20, -20, 5, 5], [500, 300, 500.4, 300.4]]   # degenerate / edge
    return data, rois


def test_roi_pool_matches_oracle(ops):
    data, rois = _roi_case(0)
    out, arg = ops.roi_pool(T(data), T(rois), return_argmax=True)
    o_ref, a_ref = RO.roi_pool(data, rois)
    np.testing.assert_array_equal(out.cpu().numpy(), o_ref)
    np.testing.assert_array_equal(arg.cpu().numpy(), a_ref)


def test_deform_psroi_pool_matches_oracle(ops):
    data, rois = _roi_case(1)
    out, cnt = ops.deform_psroi_pool(T(data), T(rois), output_dim=64, return_count=True)
    o_ref, c_ref = RO.deform_psroi_pool(data, rois, output_dim=64)
    np.testing.assert_array_equal(cnt.cpu().numpy(), c_ref)
    np.testing.assert_allclose(out.cpu().numpy(), o_ref, rtol=1e-5, atol=1e-6)
    trans = (np.random.default_rng(2).standard_normal((rois.shape[0], 2, 7, 7))).astype(np.float32)
    out, cnt = ops.deform_psroi_pool(T(data), T(rois), T(trans), output_dim=64, trans_std=0.1, return_count=True)
    o_ref, c_ref = RO.deform_psroi_pool(data, rois, trans, output_dim=64, trans_std=0.1)
    np.testing.assert_array_equal(cnt.cpu().numpy(), c_ref)
    np.testing.assert_allclose(out.cpu().numpy(), o_ref, rtol=1e-5, atol=1e-6)


def test_deform_conv_matches_oracle(ops):
    rng = np.random.default_rng(6)
    C, H, W, Co = 32, 19, 23, 48
    data = rng.standard_normal((1, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((1, 4 * 18, H, W)) * 2.0).astype(np.float32)
    wgt = (rng.standard_normal((Co, C, 3, 3)) * 0.05).astype(np.float32)
    col = ops.deform_im2col(T(data[0]), T(off[0])).cpu().numpy()
    np.testing.assert_array_equal(col, RO.deform_im2col(data[0], off[0]))
    out = ops.deform_conv(T(data), T(off), T(wgt)).cpu().numpy()
    assert rel_err(out, RO.deform_conv(data, off, wgt)) < 1e-5
    if ops.device_info()['sm100']:      # tensor-core form: fp16 transposed col buffer + tcgen05 GEMM
        out16 = ops.deform_conv(T(data), T(off), T(wgt), precision='f16').cpu().numpy()
        assert rel_err(out16, RO.deform_conv(data, off, wgt)) < 2e-3
    # zero offsets == plain dilated convolution
    out0 = ops.deform_conv(T(data), T(off * 0), T(wgt))
    torch.backends.cudnn.allow_tf32 = False
    ref0 = torch.nn.functional.conv2d(T(data), T(wgt), padding=2, dilation=2)
    assert float((out0 - ref0).abs().max() / ref0.abs().max()) < 1e-4


# ------------------------------------------------------------------------------------------------ fused head / pipeline
def test_roi_pool_fc_fast_path(ops):
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 path')
    data, rois = _roi_case(5, nroi=120, C=64)
    rng = np.random.default_rng(9)
    W = (rng.standard_normal((96, 64 * 49)) / 56).astype(np.float32); b = rng.standard_normal(96).astype(np.float32)
    pooled, _ = RO.roi_pool(data, rois)
    ref = pooled.reshape(120, -1).astype(np.float64) @ W.astype(np.float64).T + b
    for fmt in (torch.contiguous_format, torch.channels_last):
        y = ops.roi_pool_fc(T(data).contiguous(memory_format=fmt), T(rois), T(W), T(b)).cpu().numpy()
        assert rel_err(y, ref) < 1e-3


def test_hot_path_pipeline_matches_oracle(ops):
    """proposal -> ROI pool -> fc -> relation x2 -> cls/bbox -> learn_nms, CUDA vs the numpy/C oracle (one image)."""
    import relnet_b200
    from relnet_b200.pipeline import RelationHead, init_head_params
    from oracle import pipeline_np
    prm = init_head_params(3, 'cpu')
    cls_prob, bbox_pred, info = P.make_proposal_case(5)
    feat = np.maximum(np.random.default_rng(5).standard_normal((1, 256, 38, 63)), 0).astype(np.float32)
    ref = pipeline_np.head_forward({k: v.numpy() for k, v in prm.items()}, cls_prob, bbox_pred, feat, info)
    for prec in precisions(ops):
        head = RelationHead({k: v.cuda() for k, v in prm.items()}, precision=prec)
        out = head.forward(T(cls_prob), T(bbox_pred), T(feat), T(info))
        np.testing.assert_array_equal(out['rois'].cpu().numpy(), ref['rois'])
        e_feat = rel_err(out['fc_all_2_relu'].cpu().numpy(), ref['fc_all_2_relu'])
        e_cls = rel_err(out['cls_score'].cpu().numpy(), ref['cls_score'])
        e_ss = rel_err(out['sorted_score'].cpu().numpy(), ref['sorted_score'])
        fin, rfin = out['nms_final_score_output'].cpu().numpy(), ref['nms_final_score_output']
        if prec == 'fp32':
            e_fin = rel_err(fin, rfin)
        else:
            # near-tied class scores may swap ranks between fp16 and fp32 pipelines (the head is random-init: 300 rois
            # with almost equal scores per class), which permutes rows of the learn-NMS output -- compare per class
            # as sorted multisets, which is invariant to such swaps
            e_fin = rel_err(np.sort(fin, axis=0), np.sort(rfin, axis=0))
        print('pipeline[%s]: fc_all_2 %.2e cls_score %.2e sorted_score %.2e final %.2e' % (prec, e_feat, e_cls, e_ss, e_fin))
        tol = 3e-4 if prec == 'fp32' else 3e-3          # two relation modules + 4 fp16 GEMMs (K up to 12544) in sequence
        assert e_feat < tol and e_cls < tol and e_ss < tol and e_fin < (2 * tol if prec == 'fp32' else 2e-2)


def test_f16_side_channels_are_bitwise_the_same_path(ops):
    """x_f16 / want_f16 (fp16 copies handed from one layer's epilogue to the next GEMM) change launches, not results"""
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 path only')
    c = R.make_relation_case(77, 300, 1024, 16)
    t = [T(c[k]) for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]
    ref = ops.relation(*t, group=16, residual_relu=True, precision='f16')
    out, out_h = ops.relation(*t, group=16, residual_relu=True, precision='f16', x_f16=t[0].half(), want_f16=True)
    assert torch.equal(out, ref) and torch.equal(out_h, ref.half())
    W = T(np.random.RandomState(1).randn(256, 1024).astype(np.float32) * 0.03); b = T(np.zeros(256, np.float32))
    y = ops.linear(ref, W, b, precision='f16')
    y2, y2_h = ops.linear(ref, W, b, precision='f16', x_f16=out_h, want_f16=True)
    assert torch.equal(y, y2) and torch.equal(y2_h, y.half())
    with pytest.raises(Exception):
        ops.relation(*t, group=16, residual_relu=True, precision='f16', x_f16=t[0].half()[:100])


def test_linear_multi_equals_separate_layers(ops):
    """cls_score + bbox_pred + roi_feat_embedding as ONE GEMM (SURVEY 8f rank 3) == three rn_linear_packed calls"""
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 path only')
    rng = np.random.RandomState(5)
    x = T(rng.randn(300, 1024).astype(np.float32))
    layers = [(T((rng.randn(o, 1024) * 0.03).astype(np.float32)), T(rng.randn(o).astype(np.float32))) for o in (81, 8, 128)]
    x16 = x.half()
    ys = ops.linear_multi(x16, layers)
    for (W, b), y in zip(layers, ys):
        ref = ops.linear(x, W, b, precision='f16')
        assert y.shape == ref.shape and y.is_contiguous()
        assert torch.equal(y, ref)
        want = x16.float().double() @ W.half().float().double().T + b.double()
        assert rel_err(y.cpu().numpy(), want.cpu().numpy()) <= 1e-5          # fp16 operands, fp32 accumulate
    ys1 = ops.linear_multi(x16, layers[:1])
    assert torch.equal(ys1[0], ys[0])
    with pytest.raises(Exception):
        ops.linear_multi(x16, layers + layers)                               # more than 4 layers


def test_relation_fpn_form_matches_reference_execution(ops):
    """row a4 on the device: key_index (FPN non_gt_index) form against the golden made by executing the FPN symbol"""
    g = golden('relation_fpn_n90_k70')
    c = R.make_relation_case(int(g['seed']), int(g['N']), int(g['d']), int(g['H']), init='fan_in')
    t = [T(c[k]) for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]
    kidx = torch.from_numpy(g['non_gt_index'].astype(np.int32)).cuda()
    for prec in precisions(ops):
        out = ops.relation(*t, key_index=kidx, group=int(g['H']), residual_relu=False, precision=prec)
        e = rel_err(out.cpu().numpy(), g['attention'])
        print('fpn form [%s] %.2e' % (prec, e))
        assert e <= (3e-4 if prec == 'fp32' else 1e-3)


def test_learn_nms_non_gt_index_form_matches_reference_execution(ops):
    """FPN form of learn_nms (non_gt_index list + means/stds) on the device, through ops and through the CustomOp surface"""
    from relnet_b200 import compat
    g = golden('learn_nms_nongt_index')
    c = L.make_learn_nms_case(int(g['seed']), R=int(g['R']), C=int(g['C']), init='fan_in')
    w = {k: T(v) for k, v in c['P'].items()}
    idx = torch.from_numpy(g['non_gt_index'].astype(np.int32)).cuda()
    for prec in precisions(ops):
        multi, sbbox, sscore, _ = ops.learn_nms(T(c['cls_score']), T(c['bbox_pred']), T(c['rois']), T(c['im_info']), T(c['feat']),
                                                w, first_n=int(g['first_n']), means=tuple(g['means']), stds=tuple(g['stds']),
                                                non_gt_index=idx, precision=prec)
        np.testing.assert_allclose(sscore.cpu().numpy(), g['sorted_score'], rtol=2e-5, atol=1e-8)
        np.testing.assert_allclose(sbbox.cpu().numpy(), g['sorted_bbox'], rtol=1e-5, atol=2e-3)
        assert rel_err(multi.cpu().numpy(), g['nms_multi_score']) < 1e-3
    out = compat.Custom(op_type='learn_nms', num_fg_classes=int(g['C']), bbox_means='[0.0 0.0 0.0 0.0]',
                                    bbox_stds='[0.1 0.1 0.2 0.2]', first_n=int(g['first_n']), class_agnostic=True, num_thresh=5,
                                    class_thresh=0.01, nongt_dim=None, has_non_gt_index=True, cls_score=T(c['cls_score']),
                                    bbox_pred=T(c['bbox_pred']), rois=T(c['rois']), im_info=T(c['im_info']),
                                    fc_all_2_relu=T(c['feat']), non_gt_index=idx.float(), **w)
    assert rel_err(out[0].cpu().numpy(), g['nms_multi_score']) < 1e-3
