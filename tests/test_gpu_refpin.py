"""GPU: pin the C restatements (oracle/oracle_c.c) AND the product kernels of the two `operator_cxx` ops against the
REFERENCE's own CUDA kernels at the sizes the Deformable Faster-RCNN config runs them (res5 deformable conv: 512 ch, 38 x 63,
4 deformable groups; PS-ROI pooling: R = 300, 256 ch), plus an independent implementation of ROIPooling (torchvision) since
MXNet's own roi_pooling.cu is not in the reference tree.

What the reference kernels compute on these seeded inputs is stored in tests/golden/reference_deform_kernels.npz, recorded on
a B200 by tests/golden/make_reference_kernels.py from the reference's own sources (oracle/Makefile, oracle/ref_deform.cu +
oracle/ref_stub/).  Outputs of up to 11 M elements are stored as digests (conftest.digest: a seeded sample of the elements
plus sums and zero counts over 64 slices); the PS-ROI sample counts are stored whole.  A digest pins the oracle to the
reference less tightly than a full-tensor comparison: element by element only at its 1024 samples (and exactly in where the
zeros fall), elsewhere only through the slice sums, whose bound grows with the slice length.  Every element of the product
is held against the oracle.

Tolerances: sample counts bit-exact; values 1e-5 (the reference's deformable library is compiled with -fmad=false like the
oracle and the product, oracle/Makefile: the forward values agree bit for bit, the bound leaves room for last-bit
differences); atomicAdd backward 1e-5 of the tensor max (summation order differs run to run).  Product against oracle: the
sum of the two bounds.
"""
import numpy as np
import pytest
import torch
from conftest import digest_err, digest_rel_err, golden_digests, rel_err
from oracle import rois_np as RO
from oracle import relation_np as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops(cuda_device):
    import __graft_entry__ as g
    g.build()
    import relnet_b200
    torch.cuda.set_device(cuda_device)
    return relnet_b200.ops


@pytest.fixture(scope='module')
def ref():
    return golden_digests('reference_deform_kernels')


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _conv_case(seed, C=512, H=38, W=63):
    rng = np.random.default_rng(seed)
    im = rng.standard_normal((C, H, W)).astype(np.float32)
    off = (rng.standard_normal((4 * 18, H, W)) * 2.0).astype(np.float32)         # several pixels: samples leave the image
    off[:, :2] *= 8.0
    return im, off


def test_deform_im2col_reference_vs_oracle_vs_product(ops, ref):
    im, off = _conv_case(0)
    g = ref['im2col']
    orc = RO.deform_im2col(im, off)
    ours = ops.deform_im2col(T(im), T(off)).cpu().numpy()
    print('deformable im2col 512x38x63: oracle_c vs reference kernel %.2e, product vs reference kernel %.2e'
          % (digest_rel_err(orc, g), digest_rel_err(ours, g)))
    assert digest_err(orc, g, 1e-5, 1e-5) <= 1
    assert digest_err(ours, g, 1e-5, 1e-5) <= 1
    np.testing.assert_allclose(ours, orc, rtol=2e-5, atol=2e-5)
    zeros = [(p == 0).sum() for p in np.array_split(orc.ravel(), len(g['zeros']))]
    assert np.array_equal(g['val'] == 0, orc.ravel()[g['idx']] == 0) and np.array_equal(zeros, g['zeros']), \
        'out-of-image samples differ'


def _col2im_case(C=128, H=38, W=63, Co=64):                                    # backward at full spatial size, fewer channels
    rng = np.random.default_rng(3)
    data = rng.standard_normal((1, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((1, 4 * 18, H, W)) * 2.0).astype(np.float32)
    wgt = (rng.standard_normal((Co, C, 3, 3)) * 0.05).astype(np.float32)
    dout = rng.standard_normal((1, Co, H, W)).astype(np.float32)
    col = np.ascontiguousarray((wgt.reshape(Co, -1).T @ dout[0].reshape(Co, -1)).reshape(C * 9, H, W), np.float32)
    return data, off, wgt, dout, col


def test_deform_col2im_and_coord_reference_vs_oracle_vs_product(ops, ref):
    data, off, wgt, dout, col = _col2im_case()
    g_im, g_off = ref['col2im'], ref['coord']
    dd_o, doff_o, _ = RO.deform_conv_backward(dout, data, off, wgt)
    print('col2im: oracle_c vs reference %.2e | col2im_coord: oracle_c vs reference %.2e'
          % (digest_rel_err(dd_o[0], g_im), digest_rel_err(doff_o[0], g_off)))
    assert digest_rel_err(dd_o[0], g_im) < 1e-5 and digest_rel_err(doff_o[0], g_off) < 1e-5
    dd, doff, dw, _ = ops.deform_conv_backward(T(dout), T(data), T(off), T(wgt))
    dd, doff = dd.cpu().numpy()[0], doff.cpu().numpy()[0]
    assert digest_rel_err(dd, g_im) < 2e-5 and digest_rel_err(doff, g_off) < 2e-5
    assert rel_err(dd, dd_o[0]) < 3e-5 and rel_err(doff, doff_o[0]) < 3e-5


def _psroi_case(seed, R_=300, C=256, H=38, W=63):
    rng = np.random.default_rng(seed)
    data = rng.standard_normal((1, C, H, W)).astype(np.float32)
    boxes = R.make_boxes(rng, R_)
    rois = np.hstack([np.zeros((R_, 1), np.float32), boxes]).astype(np.float32)
    rois[:4, 1:] = [[0, 0, 0, 0], [990, 590, 999, 599], [-20, -20, 5, 5], [500, 300, 500.4, 300.4]]
    trans = rng.standard_normal((R_, 2, 7, 7)).astype(np.float32)
    return data, rois, trans


def _psroi_kw(with_trans):
    return dict(output_dim=256, trans_std=0.1 if with_trans else 0.0)


def _psroi_dout(shape):
    return np.random.default_rng(9).standard_normal(shape).astype(np.float32)


@pytest.mark.parametrize('with_trans', [False, True])
def test_deform_psroi_reference_vs_oracle_vs_product(ops, ref, with_trans):
    data, rois, trans = _psroi_case(1)
    tr = trans if with_trans else None
    kw = _psroi_kw(with_trans)
    p = 'psroi%d' % with_trans
    g = ref[p]
    c_ref = np.broadcast_to(g['count'][:, None].astype(np.float32), tuple(g['shape']))     # the same for every channel
    o_orc, c_orc = RO.deform_psroi_pool(data, rois, tr, **kw)
    o_our, c_our = ops.deform_psroi_pool(T(data), T(rois), T(tr) if with_trans else None, return_count=True, **kw)
    o_our = o_our.cpu().numpy()
    print('PS-ROI pool R=300 C=256 trans=%s: oracle_c vs reference %.2e, product vs reference %.2e'
          % (with_trans, digest_rel_err(o_orc, g), digest_rel_err(o_our, g)))
    np.testing.assert_array_equal(c_orc, c_ref)
    np.testing.assert_array_equal(c_our.cpu().numpy(), c_ref)
    assert digest_err(o_orc, g, 1e-5, 1e-5) <= 1
    assert digest_err(o_our, g, 1e-5, 1e-5) <= 1
    np.testing.assert_allclose(o_our, o_orc, rtol=2e-5, atol=2e-5)
    # the channels-last forms (fp32, and bf16 = the trunk's layout): same table, vector taps
    d_cl = T(data).contiguous(memory_format=torch.channels_last)
    o_cl, c_cl = ops.deform_psroi_pool(d_cl, T(rois), T(tr) if with_trans else None, return_count=True, **kw)
    o_cl = o_cl.cpu().numpy()
    np.testing.assert_array_equal(c_cl.cpu().numpy(), c_ref)
    assert digest_err(o_cl, g, 1e-5, 1e-5) <= 1
    np.testing.assert_allclose(o_cl, o_orc, rtol=2e-5, atol=2e-5)
    d_bf = d_cl.to(torch.bfloat16)
    o_bf = ops.deform_psroi_pool(d_bf, T(rois), T(tr) if with_trans else None, **kw).cpu().numpy()
    assert digest_err(o_bf, ref[p + '_bf'], 1e-5, 1e-5) <= 1
    o_orc_bf, _ = RO.deform_psroi_pool(d_bf.float().cpu().numpy(), rois, tr, **kw)
    np.testing.assert_allclose(o_bf, o_orc_bf, rtol=2e-5, atol=2e-5)
    # backward of the same op (atomicAdd: summation order differs run to run)
    dout = _psroi_dout(c_ref.shape)
    dd_orc, dt_orc = RO.deform_psroi_pool_backward(dout, c_ref, data, rois, tr, **kw)
    dd_our, dt_our = ops.deform_psroi_pool_backward(T(dout), T(c_ref), T(data), T(rois), T(tr) if with_trans else None, **kw)
    dd_our = dd_our.cpu().numpy()
    assert digest_rel_err(dd_orc, ref[p + '_dd']) < 1e-5 and digest_rel_err(dd_our, ref[p + '_dd']) < 1e-5
    assert rel_err(dd_our, dd_orc) < 2e-5
    if with_trans:
        dt_our = dt_our.cpu().numpy()
        assert digest_rel_err(dt_orc, ref[p + '_dt']) < 1e-4 and digest_rel_err(dt_our, ref[p + '_dt']) < 1e-4
        assert rel_err(dt_our, dt_orc) < 2e-4


def test_roi_pool_vs_independent_implementation(ops):
    """MXNet's ROIPooling source is not in the reference tree; torchvision.ops.roi_pool is an independent implementation of
    the same Fast R-CNN definition (round(x * scale), max(end - start + 1, 1), floor/ceil bin edges, empty bin -> 0)."""
    tv = pytest.importorskip('torchvision.ops')
    rng = np.random.default_rng(4)
    data = rng.standard_normal((1, 256, 38, 63)).astype(np.float32)
    boxes = R.make_boxes(rng, 300)
    rois = np.hstack([np.zeros((300, 1), np.float32), boxes]).astype(np.float32)
    rois[:3, 1:] = [[0, 0, 0, 0], [990, 590, 999, 599], [500, 300, 500.4, 300.4]]
    ref = tv.roi_pool(T(data), T(rois), (7, 7), 1.0 / 16).cpu().numpy()
    orc, _ = RO.roi_pool(data, rois)
    ours = ops.roi_pool(T(data), T(rois)).cpu().numpy()
    assert np.array_equal(orc, ref), 'oracle_c ROIPooling differs from torchvision roi_pool'
    assert np.array_equal(ours, ref)


def test_deform_conv_channels_last_fast_path(ops):
    """rn_deform_conv_nhwc_fwd (bf16 channels_last in, fp16 column buffer, tcgen05 GEMM, bias + relu fused) at the res5 size
    against the float32 C oracle evaluated on the same bf16-rounded data: 2e-3 of the tensor max (fp16 operands)."""
    if not ops.device_info()['sm100']:
        pytest.skip('tcgen05 needs sm_100')
    rng = np.random.default_rng(8)
    C, H, W, Co = 512, 38, 63, 512
    data = rng.standard_normal((1, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((1, 72, H, W)) * 2.0).astype(np.float32)
    wgt = (rng.standard_normal((Co, C, 3, 3)) * 0.02).astype(np.float32)
    bias = rng.standard_normal(Co).astype(np.float32)
    d_bf = T(data).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    ref = RO.deform_conv(d_bf.float().cpu().numpy(), off, wgt, bias)
    out = ops.deform_conv_nhwc(d_bf, T(off), T(wgt), T(bias), relu=False, out_dtype=torch.float32)
    assert out.is_contiguous(memory_format=torch.channels_last)
    e = rel_err(out.cpu().numpy(), ref)
    print('deformable conv 512->512 @38x63, channels_last bf16 in: rel err vs oracle %.2e' % e)
    assert e < 2e-3
    out16 = ops.deform_conv_nhwc(d_bf, T(off), T(wgt), T(bias), relu=True)
    assert rel_err(out16.float().cpu().numpy(), np.maximum(ref, 0)) < 3e-3
