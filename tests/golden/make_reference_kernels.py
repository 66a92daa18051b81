"""Record what the REFERENCE's own CUDA kernels compute on the inputs of tests/test_gpu_refpin.py and of the NMS test in
tests/test_gpu_parity.py, so that those tests compare against the reference without it.

Needs a GPU and the libraries oracle/Makefile compiles from the reference tree into oracle/_ref/ (libref_deform.so,
libref_gpu_nms.so):   python tests/golden/make_reference_kernels.py [OUTDIR]

  reference_deform_kernels.npz  deformable im2col / col2im / col2im_coord and DeformablePSROIPooling forward / backward
                                at the Deformable Faster-RCNN sizes.  Each output is stored as a digest (tests/conftest.py:
                                seeded sample of its elements, chunk sums, zeros, max), fields '<output>_<field>'; the
                                PS-ROI sample counts are stored whole, once per (roi, bin) since they do not depend on the
                                channel.
  reference_gpu_nms.npz         the keep list of lib/nms/nms_kernel.cu for the 3000 boxes of the NMS test.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)

from conftest import digest                        # noqa: E402
from oracle import rois_np as RO                   # noqa: E402
import test_gpu_refpin as RP                       # noqa: E402
import test_gpu_parity as GP                       # noqa: E402


def _put(out, key, a):
    for f, v in digest(a.cpu().numpy() if torch.is_tensor(a) else a).items():
        out['%s_%s' % (key, f)] = v


def deform(path):
    T = RP.T
    out = {}
    im, off = RP._conv_case(0)
    _put(out, 'im2col', RO.ref_deform_im2col(T(im), T(off)))
    data, off, wgt, dout, col = RP._col2im_case()
    _put(out, 'col2im', RO.ref_deform_col2im(T(col), T(off[0]), data.shape[1:]))
    _put(out, 'coord', RO.ref_deform_col2im_coord(T(col), T(data[0]), T(off[0])))
    data, rois, trans = RP._psroi_case(1)
    for with_trans in (False, True):
        p = 'psroi%d' % with_trans
        tr = T(trans) if with_trans else None
        kw = RP._psroi_kw(with_trans)
        o, c = RO.ref_deform_psroi_pool(T(data), T(rois), tr, **kw)
        c = c.cpu().numpy()
        assert (c == c[:, :1]).all() and (c == np.round(c)).all() and c.max() < 256
        out[p + '_count'] = c[:, 0].astype(np.uint8)
        _put(out, p, o)
        d_bf = T(data).contiguous(memory_format=torch.channels_last).to(torch.bfloat16)
        _put(out, p + '_bf', RO.ref_deform_psroi_pool(d_bf.float().contiguous(), T(rois), tr, **kw)[0])
        dd, dt = RO.ref_deform_psroi_pool_backward(T(RP._psroi_dout(o.shape)), T(c), T(data), T(rois), tr, **kw)
        _put(out, p + '_dd', dd)
        if with_trans:
            _put(out, p + '_dt', dt)
    np.savez_compressed(path, **out)


def nms(path):
    dets = GP._nms_case()
    np.savez_compressed(path, thresh=np.float32(0.7), keep=RO.ref_gpu_nms(dets, 0.7).astype(np.int32))


def main(outdir=HERE):
    assert RO.ref_deform_available() and RO.ref_gpu_nms_available(), 'oracle/_ref/ not built (see oracle/Makefile)'
    assert torch.cuda.is_available(), 'the reference kernels run on the GPU'
    deform(os.path.join(outdir, 'reference_deform_kernels.npz'))
    nms(os.path.join(outdir, 'reference_gpu_nms.npz'))


if __name__ == '__main__':
    main(*sys.argv[1:])
