"""GPU: the reference-facing call surfaces (compat/) drive the C ABI and reproduce the golden vectors -- these tests
read like the calls in the reference's get_symbol bodies and CustomOps."""
import numpy as np
import pytest
import torch
from conftest import golden, golden_rel_err, rel_err
from oracle import relation_np as R, learn_nms_np as L, proposal_np as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def compat(cuda_device):
    import __graft_entry__ as g
    g.build()
    import relnet_b200
    from relnet_b200 import compat
    torch.cuda.set_device(cuda_device)
    return compat


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_symbol_methods_bind_like_get_symbol(compat):
    """The body of SYM_REL:254-268 with torch tensors instead of mx symbols."""
    g = golden('relation_n300_d1024')
    c = R.make_relation_case(int(g['seed']), 300, 1024, 16, init=str(g['init']))
    params = {'pair_pos_fc1_1_weight': c['Wg'], 'pair_pos_fc1_1_bias': c['bg'], 'query_1_weight': c['Wq'],
              'query_1_bias': c['bq'], 'key_1_weight': c['Wk'], 'key_1_bias': c['bk'],
              'linear_out_1_weight': c['Wout'].reshape(1024, 1024, 1, 1), 'linear_out_1_bias': c['bout']}
    sym = compat.RelationSymbols({k: T(v) for k, v in params.items()})
    nongt_dim = 300
    sliced_rois = T(c['boxes'])
    position_matrix = sym.extract_position_matrix(sliced_rois, nongt_dim=nongt_dim)
    position_embedding = sym.extract_position_embedding(position_matrix, feat_dim=64)
    fc_new_1 = T(c['X'])
    attention_1 = sym.attention_module_multi_head(fc_new_1, position_embedding, nongt_dim=nongt_dim, fc_dim=16,
                                                  feat_dim=1024, index=1, group=16, dim=(1024, 1024, 1024))
    fc_all_1_relu = torch.relu(fc_new_1 + attention_1)
    assert golden_rel_err(attention_1.cpu().numpy(), g, 'attention') < 1e-3
    assert golden_rel_err(fc_all_1_relu.cpu().numpy(), g, 'out') < 1e-3
    # the lazy handles materialise to the reference tensors
    pm, pe = g['position_matrix'], g['position_embedding']
    np.testing.assert_allclose(position_matrix.materialize().cpu().numpy()[:len(pm)], pm, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(position_embedding.materialize().cpu().numpy()[:len(pe)], pe, atol=2e-4)
    with pytest.raises(AssertionError):
        sym.attention_module_multi_head(fc_new_1, position_embedding, nongt_dim=nongt_dim, fc_dim=8, group=16)


def test_custom_ops_protocol(compat):
    g = golden('proposal_38x63')
    cls_prob, bbox_pred, info = P.make_proposal_case(int(g['seed']))
    rois, score = compat.Custom(op_type='proposal', cls_prob=T(cls_prob), bbox_pred=T(bbox_pred), im_info=T(info),
                                feat_stride=16, scales=(4, 8, 16, 32), ratios=(0.5, 1, 2), output_score=True,
                                rpn_pre_nms_top_n=6000, rpn_post_nms_top_n=300, threshold=0.7, rpn_min_size=0)
    np.testing.assert_array_equal(score.cpu().numpy(), g['scores'])
    with pytest.raises(ValueError):
        compat.Custom(op_type='proposal', cls_prob=T(np.tile(cls_prob, (2, 1, 1, 1))), bbox_pred=T(np.tile(bbox_pred, (2, 1, 1, 1))),
                      im_info=T(info), rpn_post_nms_top_n=300)

    gt = golden('proposal_target_300_7')
    cfg = dict(CLASS_AGNOSTIC=True, TRAIN=dict(BG_THRESH_HI=0.5, BBOX_NORMALIZATION_PRECOMPUTED=True,
                                               BBOX_MEANS=[0.0] * 4, BBOX_STDS=[0.1, 0.1, 0.2, 0.2], BBOX_WEIGHTS=[1.0] * 4))
    r, lab, bt, bw = compat.Custom(op_type='proposal_target', rois=T(gt['rois']), gt_boxes=T(gt['gt_boxes']),
                                   num_classes=2, batch_images=1, batch_rois=-1, cfg=cfg, fg_fraction=0.25)
    np.testing.assert_array_equal(lab.cpu().numpy(), gt['label'])
    np.testing.assert_allclose(bt.cpu().numpy(), gt['bbox_target'], rtol=2e-6, atol=2e-6)

    gl = golden('learn_nms_r60_c8')
    c = L.make_learn_nms_case(int(gl['seed']), R=60, C=8, init=str(gl['init']))
    prop = compat.LearnNmsProp(num_fg_classes='8', bbox_means='None', bbox_stds='None', first_n='30', class_agnostic='True',
                               num_thresh='5', class_thresh='0.01', nongt_dim='60', has_non_gt_index='False')
    assert prop.list_arguments()[:5] == ['cls_score', 'bbox_pred', 'rois', 'im_info', 'fc_all_2_relu']
    vals = dict(cls_score=c['cls_score'], bbox_pred=c['bbox_pred'], rois=c['rois'], im_info=c['im_info'],
                fc_all_2_relu=c['feat'], **c['P'])
    in_data = [T(vals[k]) for k in prop.list_arguments()]
    _, out_shapes = prop.infer_shape([tuple(t.shape) for t in in_data])
    out_data = [torch.zeros(s, device='cuda') for s in out_shapes]
    op = prop.create_operator(None, None, None)
    op.forward(False, ['write'] * 3, in_data, out_data, [])
    assert rel_err(out_data[0].cpu().numpy(), gl['nms_multi_score']) < 1e-3
    np.testing.assert_allclose(out_data[2].cpu().numpy(), gl['sorted_score'], rtol=2e-5)
    assert rel_err(op.nms_final_score.cpu().numpy(), gl['final_score']) < 1e-3
    grads = [torch.ones_like(t) for t in in_data]
    op.backward(['write'] * len(grads), None, in_data, out_data, grads, [])
    assert all(float(gd.abs().sum()) == 0 for gd in grads)          # the reference op returns zero gradients


def test_c_symbol_replacements(compat):
    rng = np.random.default_rng(3)
    boxes = R.make_boxes(rng, 500); sc = rng.permutation(500).astype(np.float32) / 500
    dets = np.hstack([boxes, sc[:, None]]).astype(np.float32)
    assert compat.gpu_nms(dets, 0.7) == P.gpu_nms(dets, 0.7)
    ov = compat.bbox_overlaps_cython(boxes[:50].astype(np.float64), boxes[50:60].astype(np.float64))
    np.testing.assert_allclose(ov, P.bbox_overlaps(boxes[:50], boxes[50:60]), rtol=1e-14)


def test_box_annotator_ohem_custom_op(compat):
    """mx.sym.Custom(op_type='BoxAnnotatorOHEM', ...) call form (SYM_REL:299-305) against the reference-executed golden"""
    g = golden('box_annotator_ohem')
    dev = lambda k: torch.from_numpy(g[k]).cuda()
    lab, w = compat.Custom(op_type='BoxAnnotatorOHEM', num_classes=81, num_reg_classes=2, roi_per_img=128,
                                       cls_score=dev('cls_score'), bbox_pred=dev('bbox_pred'), labels=dev('labels'),
                                       bbox_targets=dev('bbox_targets'), bbox_weights=dev('bbox_weights'))
    assert np.array_equal(lab.cpu().numpy(), g['labels_ohem']) and np.array_equal(w.cpu().numpy(), g['bbox_weights_ohem'])


def test_streaming_detector_matches_single_image_path(compat):
    """pipeline.StreamingDetector (2 slots in flight, copies on side streams) returns, image by image, exactly what the
    one-image-at-a-time graph replay returns"""
    import relnet_b200
    from relnet_b200.pipeline import RelationHead, init_head_params, Detector, GraphedStep, StreamingDetector
    from relnet_b200.trunk import make_trunk
    dev = torch.device('cuda')
    trunk = make_trunk(dev, torch.bfloat16)
    head = RelationHead(init_head_params(0, dev), precision='f16' if relnet_b200.ops.device_info()['sm100'] else 'fp32')
    im_info = torch.tensor([[224.0, 320.0, 1.0]], device=dev)
    imgs = [(torch.randn(1, 3, 224, 320, generator=torch.Generator().manual_seed(s)) * 50).pin_memory() for s in range(5)]
    single = GraphedStep(Detector(trunk, head, im_info), [imgs[0].to(dev)])
    want = []
    for im in imgs:
        o = single(im.to(dev))
        torch.cuda.synchronize()
        want.append({k: o[k].cpu().clone() for k in StreamingDetector.OUT})
    sd = StreamingDetector(trunk, head, im_info, imgs[0].to(dev), depth=2)
    got, tickets = [], []
    for im in imgs:
        tickets.append(sd.submit(im))
        if len(tickets) == 2:
            got.append({k: v.clone() for k, v in sd.collect(tickets.pop(0)).items()})
    while tickets:
        got.append({k: v.clone() for k, v in sd.collect(tickets.pop(0)).items()})
    assert len(got) == len(want)
    for g, w in zip(got, want):
        for k in StreamingDetector.OUT:
            assert torch.equal(g[k], w[k]), k
    with pytest.raises(RuntimeError):
        sd.submit(imgs[0]); sd.submit(imgs[1]); sd.submit(imgs[2])        # third submit without a collect: slot busy
