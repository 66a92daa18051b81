"""The operator boundary schema: the compat CustomOpProp classes must answer exactly what the REFERENCE's own Prop classes answer
(executed from /root/reference by tests/golden/make_prop_schema.py -> tests/golden/prop_schema.json) for the string kwargs MXNet
hands a CustomOpProp: registered op_type, argument / output names and order, need_top_grad, inferred shapes, parsed attributes.
No device work: Prop classes are host-only."""
import json
import os
import pickle

import numpy as np
import pytest

import relnet_b200  # noqa: F401  (package alias)
from relnet_b200.compat import operators as C

HERE = os.path.dirname(os.path.abspath(__file__))
G = json.load(open(os.path.join(HERE, 'golden', 'prop_schema.json')))


def _norm(x):
    if isinstance(x, (list, tuple)):
        return [_norm(v) for v in x]
    if isinstance(x, np.ndarray):
        return _norm(x.tolist())
    if isinstance(x, (bool, str, type(None))):
        return x
    if isinstance(x, float):
        return x if x != int(x) else int(x)
    return int(x)


@pytest.mark.parametrize('case', G['cases'], ids=lambda c: '%s-%s' % (c['op_type'], c['kwargs'].get('has_non_gt_index', c['kwargs'].get('batch_rois', c['kwargs'].get('output_score', '')))))
def test_prop_matches_the_reference_prop(case):
    assert case['registered_in_reference']
    cls = C.REGISTRY[case['op_type']]                     # same op_type string as mx.operator.register(...) in the reference
    assert cls.__name__ == case['class']
    kw = dict(case['kwargs'])
    if kw.get('cfg') == '<pickle>':
        kw['cfg'] = pickle.dumps(G['cfg'])                # the reference passes cPickle.dumps(cfg) (SYM_REL:241-247)
    prop = cls(**kw)
    ref = case['reference']
    assert list(prop.list_arguments()) == ref['list_arguments']
    assert list(prop.list_outputs()) == ref['list_outputs']
    assert bool(prop.need_top_grad) == ref['need_top_grad']
    assert prop.declare_backward_dependency([], [], []) == []
    if 'infer_shape' in ref:
        got = prop.infer_shape([list(s) for s in case['in_shape']])
        assert _norm(got[:2]) == ref['infer_shape']
    for k, v in ref['attrs'].items():                     # every scalar / array attribute the reference's Prop parsed
        assert hasattr(prop, k), k
        assert _norm(getattr(prop, k)) == v, (k, getattr(prop, k), v)


def test_learn_nms_prop_refuses_comma_separated_box_statistics_like_the_reference():
    # learn_nms.py:416-417: "gluon customops use , to separate elements, make sure this doesn't happen"
    with pytest.raises(AssertionError):
        C.REGISTRY['learn_nms'](num_fg_classes='80', bbox_means='[0., 0., 0., 0.]', bbox_stds='[0.1 0.1 0.2 0.2]', first_n='100',
                                class_agnostic='False', num_thresh='5', class_thresh='0.01', nongt_dim='300', has_non_gt_index='False')


def test_proposal_prop_checks_roi_count_like_the_reference():
    with pytest.raises(AssertionError):
        C.REGISTRY['proposal']().infer_shape([[1, 24, 38, 63], [2, 48, 38, 63], [1, 3]])


# ------------------------------------------------------------------------------------------------ symbol-class methods
@pytest.mark.parametrize('symfile', sorted(G['symbol_signatures']))
def test_symbol_methods_take_the_reference_arguments(symfile):
    """Same names in the same order with the same defaults as the reference's methods (SYM_REL / SYM_REL_NMS / SYM_FPN_REL_NMS);
    the compat methods may add keywords after them and may give a default where the reference has none.  The one slot the
    reference spells two ways (nongt_dim | non_gt_index) is one slot here as well."""
    import inspect
    from relnet_b200.compat.symbols import RelationSymbols
    for fn, ref in G['symbol_signatures'][symfile].items():
        ps = list(inspect.signature(getattr(RelationSymbols, fn)).parameters.items())
        assert len(ps) >= len(ref), fn
        for (name, q), (rname, rdefault, has_default) in zip(ps, ref):
            assert name == rname or (name, rname) == ('nongt_dim', 'non_gt_index'), (fn, name, rname)
            if has_default:
                assert q.default is not inspect.Parameter.empty and _norm(q.default) == rdefault, (fn, name, q.default, rdefault)


def test_position_matrix_accepts_both_spellings_of_the_key_slot():
    import torch
    from relnet_b200.compat.symbols import RelationSymbols
    boxes = torch.zeros(10, 4)
    idx = torch.arange(6)
    a = RelationSymbols.extract_position_matrix(boxes, 7)                              # SYM_REL:52  (bbox, nongt_dim)
    assert a.nongt_dim == 7 and a.non_gt_index is None
    b = RelationSymbols.extract_position_matrix(boxes, idx)                            # SYM_FPN_REL_NMS:860  (bbox, non_gt_index)
    assert b.nongt_dim is None and b.non_gt_index is idx
    c = RelationSymbols.extract_position_matrix(boxes, non_gt_index=idx)
    assert c.nongt_dim is None and c.non_gt_index is idx
    d = RelationSymbols.extract_position_matrix(boxes, nongt_dim=np.int64(7))          # numpy scalars are counts, not index lists
    assert int(d.nongt_dim) == 7 and d.non_gt_index is None
    e = RelationSymbols.extract_position_embedding(b, 64)
    assert e.pm is b and e.feat_dim == 64 and e.wave_length == 1000


@pytest.mark.parametrize('op', sorted(G['cxx_params']))
def test_cxx_operator_keywords_are_the_dmlc_parameter_fields(op):
    """compat.DeformableConvolution / DeformablePSROIPooling take every field of the reference's dmlc::Parameter struct
    (deformable_convolution-inl.h:39-76, deformable_psroi_pooling-inl.h:32-54) as a keyword, with the declared default where
    there is one (an empty TShape() default means stride / dilate 1, pad 0 -- MXNet's convention)."""
    import inspect
    fn = getattr(C, op)
    ps = inspect.signature(fn).parameters
    has_kw = any(q.kind is inspect.Parameter.VAR_KEYWORD for q in ps.values())
    shape_defaults = {'stride': (1, 1), 'dilate': (1, 1), 'pad': (0, 0)}
    for name, default in G['cxx_params'][op]:
        if name not in ps:
            assert has_kw and name in ('workspace', 'layout'), (op, name)      # accepted and ignored (no meaning for this library)
            continue
        if default is None:
            continue
        got = ps[name].default
        if default == 'TShape()':
            assert tuple(got) == shape_defaults[name], (op, name, got)
        elif default in ('true', 'false'):
            assert got is (default == 'true'), (op, name, got)
        else:
            assert float(got) == float(default), (op, name, got)
