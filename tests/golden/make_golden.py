"""Generate the golden vectors under tests/golden/ by EXECUTING THE REFERENCE'S OWN PYTHON.

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py

The reference (Python 2 / MXNet 1.1.0) is loaded from where it lies by oracle/refexec.py (in-memory py2->py3
transform, numpy stand-in for the MXNet ops: oracle/mxshim.py).  Inputs come from the seeded generators in oracle/*.
Each .npz stores inputs and the reference outputs; tests/test_oracle_golden.py checks the oracle restatement
against them (CPU, no GPU), tests/test_*_gpu.py check the CUDA path against them on the GPU box.

What is and is not pinned by this (also in DESIGN.md):
  * composition logic of the relation module, learn_nms op, proposal op, proposal_target op: reference code.
  * MXNet op semantics (mxshim) and the GPU NMS / cython IoU stand-ins: restatements (see refexec.py docstring).
"""
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import refexec, relation_np, learn_nms_np, proposal_np   # noqa: E402


def checksum(d):
    """Order-independent float64 checksum of every array in a case dict (detects generator drift)."""
    tot = 0.0
    for k in sorted(d):
        v = d[k]
        if isinstance(v, np.ndarray):
            a = v.astype(np.float64).ravel()
            tot += float(np.abs(a).sum()) + 1e-3 * float((a * np.arange(1, a.size + 1) % 7).sum())
    return tot


def relation_case(ns, name, seed, N, d, H, init, M=None, keep_rows=None):
    mx, shim = ns.mx, ns.mxshim
    c = relation_np.make_relation_case(seed, N, d, H, init=init, M=M)
    Sym = ns.sym_rel.resnet_v1_101_rcnn_attention_1024_pairwise_position_multi_head_16
    sym = Sym()
    M_ = M or N
    shim.PARAMS.clear()
    shim.PARAMS.update({
        'pair_pos_fc1_1_weight': c['Wg'], 'pair_pos_fc1_1_bias': c['bg'],
        'query_1_weight': c['Wq'], 'query_1_bias': c['bq'],
        'key_1_weight': c['Wk'], 'key_1_bias': c['bk'],
        'linear_out_1_weight': c['Wout'].reshape(d, d, 1, 1), 'linear_out_1_bias': c['bout']})
    pm = Sym.extract_position_matrix(shim.ND(c['boxes']), nongt_dim=M_)
    pe = Sym.extract_position_embedding(pm, feat_dim=64)
    att = sym.attention_module_multi_head(shim.ND(c['X']), pe, nongt_dim=M_, fc_dim=H, feat_dim=d,
                                          index=1, group=H, dim=(d, d, d))
    out = np.maximum(c['X'] + att.a, 0).astype(np.float32)        # fc_all = fc_new + attention; relu (SYM_REL:267-268)
    res = dict(position_embedding=pe.a[:8], attention=att.a, out=out)
    if keep_rows:
        # a seeded subset of whole rows keeps the file under 1 MB; the full tensors' maxima keep rel_err's normaliser
        rows = np.sort(np.random.default_rng(seed).choice(N, keep_rows, replace=False)).astype(np.int32)
        res = dict(position_embedding=pe.a[:1], rows=rows, attention=att.a[rows], out=out[rows],
                   attention_absmax=np.abs(att.a).max(), out_absmax=np.abs(out).max())
    # inputs are regenerated from the seed by oracle.relation_np.make_relation_case (checksum guards drift)
    np.savez_compressed(os.path.join(HERE, name + '.npz'), N=N, d=d, H=H, M=M_, init=init, seed=seed,
                        input_checksum=checksum(c),
                        position_matrix=pm.a if N <= 128 else pm.a[:8], **res)
    print(name, 'attention', att.a.shape, float(np.abs(att.a).max()))


def relation_fpn_case(ns, name, seed, N, d, H, n_keys):
    """FPN form (SYM_FPN_REL_NMS:843-977): keys = take(roi_feat, non_gt_index), pair FC as a 1x1 Convolution over the
    [1, 64, N, M] embedding (:1122-1135 shows how get_symbol prepares it)."""
    shim = ns.mxshim
    c = relation_np.make_relation_case(seed, N, d, H, init='fan_in')
    rng = np.random.default_rng(seed + 1000)
    idx = np.sort(rng.permutation(N)[:n_keys]).astype(np.float32)            # MXNet indices are float-valued
    Sym = ns.sym_fpn_rel_nms.resnet_v1_101_rcnn_fpn_attention_1024_pairwise_position_multi_head_16_learn_nms
    sym = Sym()
    shim.PARAMS.clear()
    shim.PARAMS.update({
        'pair_pos_fc1_1_weight': c['Wg'].reshape(H, 64, 1, 1), 'pair_pos_fc1_1_bias': c['bg'],
        'query_1_weight': c['Wq'], 'query_1_bias': c['bq'],
        'key_1_weight': c['Wk'], 'key_1_bias': c['bk'],
        'linear_out_1_weight': c['Wout'].reshape(d, d, 1, 1), 'linear_out_1_bias': c['bout']})
    pm = Sym.extract_position_matrix(shim.ND(c['boxes']), non_gt_index=shim.ND(idx))
    pe = Sym.extract_position_embedding(pm, feat_dim=64)
    pe_r = shim.expand_dims(shim.transpose(pe, axes=(2, 0, 1)), axis=0)
    att = sym.attention_module_multi_head(shim.ND(c['X']), pe_r, non_gt_index=shim.ND(idx), fc_dim=H, feat_dim=d,
                                          index=1, group=H, dim=(d, d, d))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), N=N, d=d, H=H, seed=seed, input_checksum=checksum(c),
                        non_gt_index=idx.astype(np.int32), position_matrix=pm.a[:8], attention=att.a)
    print(name, 'attention', att.a.shape, float(np.abs(att.a).max()))


def learn_nms_case(ns, name, seed, R, C, init, first_n):
    shim = ns.mxshim
    c = learn_nms_np.make_learn_nms_case(seed, R=R, C=C, init=init)
    prop = ns.learn_nms.LearnNmsProp(num_fg_classes=str(C), bbox_means='None', bbox_stds='None',
                                     first_n=str(first_n), class_agnostic='True', num_thresh='5',
                                     class_thresh='0.01', nongt_dim=str(R), has_non_gt_index='False')
    op = prop.create_operator(None, None, None)
    names = prop.list_arguments()
    P = c['P']
    vals = dict(cls_score=c['cls_score'], bbox_pred=c['bbox_pred'], rois=c['rois'], im_info=c['im_info'],
                fc_all_2_relu=c['feat'], **P)
    in_data = [shim.ND(vals[k]) for k in names]
    _, out_shapes = prop.infer_shape([v.shape for v in in_data])
    out_data = [shim.ND(np.zeros(s, np.float32)) for s in out_shapes]
    op.forward(False, ['write'] * 3, in_data, out_data, [])
    multi, sbbox, sscore = (o.a for o in out_data)
    final = multi.mean(axis=2, dtype=np.float32)                  # SYM_REL_NMS:553-554, MERGE_METHOD=-1
    np.savez_compressed(os.path.join(HERE, name + '.npz'), R=R, C=C, first_n=first_n, init=init, seed=seed,
                        input_checksum=checksum(dict(c, **P)),
                        nms_multi_score=multi, sorted_bbox=sbbox, sorted_score=sscore, final_score=final)
    print(name, 'multi', multi.shape, float(multi.max()), 'nonzero classes', int((multi.max(axis=(0, 2)) > 0).sum()))


def learn_nms_nongt_case(ns, name, seed, R, C, first_n, n_keep):
    """FPN form of the op: has_non_gt_index=True, the 20th input is the index list (LNMS:260-283), train-time means/stds"""
    shim = ns.mxshim
    c = learn_nms_np.make_learn_nms_case(seed, R=R, C=C, init='fan_in')
    rng = np.random.default_rng(seed + 500)
    idx = np.sort(rng.permutation(R)[:n_keep]).astype(np.float32)
    prop = ns.learn_nms.LearnNmsProp(num_fg_classes=str(C), bbox_means='[0.0 0.0 0.0 0.0]', bbox_stds='[0.1 0.1 0.2 0.2]',
                                     first_n=str(first_n), class_agnostic='True', num_thresh='5', class_thresh='0.01',
                                     nongt_dim='None', has_non_gt_index='True')
    op = prop.create_operator(None, None, None)
    names = prop.list_arguments()
    vals = dict(cls_score=c['cls_score'], bbox_pred=c['bbox_pred'], rois=c['rois'], im_info=c['im_info'],
                fc_all_2_relu=c['feat'], non_gt_index=idx, **c['P'])
    in_data = [shim.ND(vals[k]) for k in names]
    _, out_shapes = prop.infer_shape([v.shape for v in in_data])
    out_data = [shim.ND(np.zeros(s, np.float32)) for s in out_shapes]
    op.forward(False, ['write'] * 3, in_data, out_data, [])
    multi, sbbox, sscore = (o.a for o in out_data)
    np.savez_compressed(os.path.join(HERE, name + '.npz'), R=R, C=C, first_n=first_n, seed=seed, non_gt_index=idx.astype(np.int32),
                        means=np.zeros(4, np.float32), stds=np.array([0.1, 0.1, 0.2, 0.2], np.float32),
                        input_checksum=checksum(dict(c, **c['P'])), nms_multi_score=multi, sorted_bbox=sbbox, sorted_score=sscore)
    print(name, 'multi', multi.shape, float(multi.max()), 'args', len(names))


def proposal_case(ns, name, seed, H, W, im_info, pre, post, scales=(4, 8, 16, 32)):
    shim = ns.mxshim
    A = 3 * len(scales)
    cls_prob, bbox_pred, info = proposal_np.make_proposal_case(seed, H=H, W=W, A=A, im_info=im_info)
    op = ns.proposal.ProposalOperator(16, str(tuple(scales)), '(0.5, 1, 2)', True, pre, post, 0.7, 0)
    in_data = [shim.ND(cls_prob), shim.ND(bbox_pred), shim.ND(info)]
    out_data = [shim.ND(np.zeros((post, 5), np.float32)), shim.ND(np.zeros((post, 1), np.float32))]
    np.random.seed(0)
    op.forward(False, ['write', 'write'], in_data, out_data, [])
    anchors = ns.generate_anchor.generate_anchors(base_size=16, scales=np.array(scales, dtype=float),
                                                  ratios=np.array([0.5, 1, 2]))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), seed=seed, H=H, W=W, im_info=info,
                        input_checksum=checksum(dict(a=cls_prob, b=bbox_pred)),
                        pre=pre, post=post, scales=np.array(scales), rois=out_data[0].a, scores=out_data[1].a,
                        anchors=anchors)
    print(name, 'rois', out_data[0].a.shape, out_data[0].a[:2])


def proposal_target_case(ns, name, seed, N, G):
    shim = ns.mxshim
    rng = np.random.default_rng(seed)
    boxes = relation_np.make_boxes(rng, N)
    gt = relation_np.make_boxes(rng, G)
    # make some rois overlap the gt strongly so that fg labels exist
    for i in range(min(N // 4, 4 * G)):
        j = i % G
        boxes[i] = gt[j] + rng.normal(0, 6, 4).astype(np.float32)
    boxes[:, 2] = np.maximum(boxes[:, 2], boxes[:, 0] + 1); boxes[:, 3] = np.maximum(boxes[:, 3], boxes[:, 1] + 1)
    rois = np.hstack([np.zeros((N, 1), np.float32), boxes]).astype(np.float32)
    gt5 = np.hstack([gt, rng.integers(1, 81, (G, 1)).astype(np.float32)]).astype(np.float32)
    cfg = ns.EasyDict(CLASS_AGNOSTIC=True,
                      TRAIN=dict(BG_THRESH_HI=0.5, BBOX_NORMALIZATION_PRECOMPUTED=True, BBOX_MEANS=[0.0, 0.0, 0.0, 0.0],
                                 BBOX_STDS=[0.1, 0.1, 0.2, 0.2], BBOX_WEIGHTS=np.array([1.0, 1.0, 1.0, 1.0])))
    op = ns.proposal_target.ProposalTargetOperator(2, 1, -1, cfg, 0.25)
    in_data = [shim.ND(rois), shim.ND(gt5)]
    out_data = [shim.ND(np.zeros((N + G, 5), np.float32)), shim.ND(np.zeros((N + G,), np.float32)),
                shim.ND(np.zeros((N + G, 8), np.float32)), shim.ND(np.zeros((N + G, 8), np.float32))]
    op.forward(True, ['write'] * 4, in_data, out_data, [])
    ov = ns.bbox_transform.bbox_overlaps_py(rois[:, 1:].astype(np.float64), gt5[:, :4].astype(np.float64))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), rois=rois, gt_boxes=gt5, rois_out=out_data[0].a,
                        label=out_data[1].a, bbox_target=out_data[2].a, bbox_weight=out_data[3].a,
                        overlaps_py=ov)
    print(name, 'fg', int((out_data[1].a > 0).sum()), 'of', N + G)


def nms_multi_target_case(ns, name):
    """learn-NMS training labels: NmsMultiTargetOp.forward (operator_py/nms_multi_target.py:24-74)"""
    shim = ns.mxshim
    rng = np.random.default_rng(41)
    n, C, G = 100, 8, 9
    boxes = relation_np.make_boxes(rng, n * C).reshape(n, C, 4)
    gt = relation_np.make_boxes(rng, G)
    cls = rng.integers(1, C + 1, G).astype(np.float32)
    cls[:2] = 3
    for g in range(G):                     # several boxes of the right class overlap every gt
        c = int(cls[g]) - 1
        for k in range(6):
            boxes[(g * 7 + k) % n, c] = gt[g] + rng.normal(0, 4 + 3 * k, 4)
    boxes[..., 2] = np.maximum(boxes[..., 2], boxes[..., 0] + 1); boxes[..., 3] = np.maximum(boxes[..., 3], boxes[..., 1] + 1)
    boxes = boxes.astype(np.float32)
    gt5 = np.hstack([gt, cls[:, None]]).astype(np.float32)[None]
    score = rng.random((n, C)).astype(np.float32)
    th = np.array([0.5, 0.6, 0.7, 0.8, 0.9])
    op = ns.nms_multi_target.NmsMultiTargetProp('[0.5 0.6 0.7 0.8 0.9]').create_operator(None, None, None)
    out = [shim.ND(np.zeros((n, C, 5), np.float32))]
    op.forward(True, ['write'], [shim.ND(boxes), shim.ND(gt5), shim.ND(score)], out, [])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), bbox=boxes, gt_box=gt5, score=score, target_thresh=th,
                        target=out[0].a)
    print(name, 'positives', int(out[0].a.sum()))


def ohem_case(ns, name):
    """BoxAnnotatorOHEMOperator.forward (operator_py/box_annotator_ohem.py:26-53) under the numpy MXNet shim"""
    shim = ns.mxshim
    rng = np.random.default_rng(51)
    R, NC, K = 307, 81, 2
    cls_score = (rng.standard_normal((R, NC)) * 2).astype(np.float32)
    labels = np.where(rng.random(R) < 0.25, rng.integers(1, NC, R), 0).astype(np.float32)
    bbox_pred = (rng.standard_normal((R, 4 * K)) * 0.5).astype(np.float32)
    bbox_targets = np.zeros((R, 4 * K), np.float32); bbox_weights = np.zeros((R, 4 * K), np.float32)
    fg = labels > 0
    bbox_targets[fg, 4:] = (rng.standard_normal((int(fg.sum()), 4)) * 1.5).astype(np.float32)
    bbox_weights[fg, 4:] = 1
    cls_score[5] = cls_score[6]; labels[5] = labels[6] = 0          # an exact loss tie among background rois
    op = ns.box_annotator_ohem.BoxAnnotatorOHEMProp('81', '2', '128').create_operator(None, None, None)
    out = [shim.ND(np.zeros(R, np.float32)), shim.ND(np.zeros((R, 4 * K), np.float32))]
    op.forward(True, ['write', 'write'], [shim.ND(cls_score), shim.ND(bbox_pred), shim.ND(labels.copy()),
                                          shim.ND(bbox_targets), shim.ND(bbox_weights)], out, [])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), cls_score=cls_score, bbox_pred=bbox_pred, labels=labels,
                        bbox_targets=bbox_targets, bbox_weights=bbox_weights, roi_per_img=128,
                        labels_ohem=out[0].a, bbox_weights_ohem=out[1].a)
    print(name, 'kept', int((out[0].a >= 0).sum()))


def misc_case(ns, name):
    """Small pure-python reference helpers: refine_bbox_nd, rank embedding, multi position matrix, decode/encode."""
    shim = ns.mxshim
    rng = np.random.default_rng(7)
    boxes = relation_np.make_boxes(rng, 40)
    deltas = (rng.standard_normal((40, 4)) * 0.2).astype(np.float32)
    info = np.array([[600, 1000, 1.0]], np.float32)
    refined = ns.learn_nms.refine_bbox_nd(shim.ND(boxes), shim.ND(deltas), shim.ND(info)).a
    refined_ms = ns.learn_nms.refine_bbox_nd(shim.ND(boxes), shim.ND(deltas), shim.ND(info),
                                             means=np.array([0.0, 0.0, 0.0, 0.0]), stds=np.array([0.1, 0.1, 0.2, 0.2])).a
    rank = ns.learn_nms.extract_rank_embedding_nd(100, 1024).a
    sb = np.stack([boxes[:20], boxes[20:]], axis=1)                        # [n=20, C=2, 4]
    mpm = ns.learn_nms.extract_multi_position_matrix_nd(shim.ND(sb)).a     # [C,n,n,4]
    dec = ns.bbox_transform.nonlinear_pred(boxes.astype(np.float64), deltas)
    enc = ns.bbox_transform.nonlinear_transform(boxes, boxes[::-1].copy())
    np.savez_compressed(os.path.join(HERE, name + '.npz'), boxes=boxes, deltas=deltas, im_info=info,
                        refined=refined, refined_ms=refined_ms, rank_embedding=rank, sorted_bbox=sb,
                        multi_position_matrix=mpm, decoded=dec, encoded=enc)
    print(name, 'ok')


def main():
    assert refexec.available(), 'needs /root/reference'
    ns = refexec.load_reference()
    relation_case(ns, 'relation_cfg0_ref', 0, 100, 256, 4, 'ref')            # BASELINE.json configs[0], reference init
    relation_case(ns, 'relation_cfg0_fanin', 1, 100, 256, 4, 'fan_in')       # configs[0], O(1) logits
    relation_case(ns, 'relation_n300_d1024', 2, 300, 1024, 16, 'fan_in', keep_rows=24)   # the headline shape
    relation_case(ns, 'relation_n120_m100', 3, 120, 256, 4, 'fan_in', M=100)  # train-time N = M + G (nongt slice)
    learn_nms_case(ns, 'learn_nms_r300_c80', 11, 300, 80, 'fan_in', 100)
    learn_nms_case(ns, 'learn_nms_r60_c8', 12, 60, 8, 'ref', 30)
    proposal_case(ns, 'proposal_38x63', 21, 38, 63, (600.0, 1000.0, 1.0), 6000, 300)
    proposal_case(ns, 'proposal_small', 22, 10, 12, (160.0, 200.0, 1.0), 200, 32, scales=(8, 16))
    proposal_target_case(ns, 'proposal_target_300_7', 31, 300, 7)
    misc_case(ns, 'misc_helpers')
    nms_multi_target_case(ns, 'nms_multi_target')
    ohem_case(ns, 'box_annotator_ohem')
    relation_fpn_case(ns, 'relation_fpn_n90_k70', 5, 90, 256, 4, 70)
    learn_nms_nongt_case(ns, 'learn_nms_nongt_index', 13, 80, 8, 30, 64)


if __name__ == '__main__':
    main()
