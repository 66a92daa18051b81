import os
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False))


def checksum(d):
    """Same as tests/golden/make_golden.py:checksum -- guards the seeded generators against drift."""
    tot = 0.0
    for k in sorted(d):
        v = d[k]
        if isinstance(v, np.ndarray):
            a = v.astype(np.float64).ravel()
            tot += float(np.abs(a).sum()) + 1e-3 * float((a * np.arange(1, a.size + 1) % 7).sum())
    return tot


def rel_err(a, b):
    """max|a-b| / max|b| -- the per-tensor metric the 1e-3 relation tolerance is stated in (DESIGN.md)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def golden_rel_err(a, g, key):
    """rel_err of a full output `a` against the relation fixture's g[key].  A fixture that holds only a seeded subset of
    rows (g['rows']) stores the full tensor's max|ref| as g[key + '_absmax']: the figure is then rel_err over those rows,
    with the normaliser of the full tensor."""
    if 'rows' not in g:
        return rel_err(a, g[key])
    a = np.asarray(a, np.float64)[g['rows']]
    return float(np.abs(a - g[key]).max() / float(g[key + '_absmax']))


def elem_err(a, b, rtol=1e-3, atol_frac=1e-3):
    """Elementwise companion of rel_err: an element passes when |a-b| <= rtol*|b| + atol, atol = atol_frac * rms(b).
    Returns (fraction of elements violating, worst |a-b| / (rtol*|b| + atol)).  Reported beside rel_err in the f16 parity
    tests (VERDICT r1 / ADVICE: the per-tensor norm alone hides small-magnitude outputs)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    atol = atol_frac * float(np.sqrt(np.mean(b * b)) + 1e-30)
    ratio = np.abs(a - b) / (rtol * np.abs(b) + atol)
    return float(np.mean(ratio > 1.0)), float(ratio.max())


def digest(a, k=1024, chunks=64, seed=0):
    """Compact stand-in for a tensor too large to store under tests/golden/: its shape and largest magnitude, its values
    at k seeded positions, and the float64 sum, absolute sum and count of zeros of each of `chunks` equal slices of the
    flat array (so every element still enters the comparison).  It is a weaker pin than the full tensor: elements are
    compared one by one only at the samples; elsewhere an error shows only through its slice's sum."""
    a = np.asarray(a, np.float32)
    f = a.ravel()
    idx = np.sort(np.random.default_rng(seed).choice(f.size, min(k, f.size), replace=False)).astype(np.int32)
    parts = np.array_split(f.astype(np.float64), chunks)
    return dict(shape=np.array(a.shape, np.int64), max=np.float64(np.abs(f).max()), idx=idx, val=f[idx],
                sum=np.array([p.sum() for p in parts]), abs=np.array([np.abs(p).sum() for p in parts]),
                zeros=np.array([(p == 0).sum() for p in parts], np.int64))


def digest_err(x, d, rtol, atol):
    """Worst |x - ref| / (atol + rtol |ref|) over the digest's sampled elements and its chunk sums, where the bound of a sum
    is the sum of its elements' bounds: <= 1 wherever np.allclose(x, ref, rtol, atol) holds on the full tensor.
    With rtol = 0 and atol = eps * max|ref| it is <= 1 wherever rel_err(x, ref) <= eps."""
    x = np.asarray(x, np.float64)
    assert x.shape == tuple(d['shape']), (x.shape, d['shape'])
    f = x.ravel()
    e = np.abs(f[d['idx']] - d['val']) / (atol + rtol * np.abs(d['val'].astype(np.float64)))
    parts = np.array_split(f, len(d['sum']))
    n = np.array([p.size for p in parts])
    s = np.abs(np.array([p.sum() for p in parts]) - d['sum']) / (atol * n + rtol * d['abs'])
    return float(max(e.max(), s.max()))


def digest_rel_err(x, d):
    """rel_err(x, ref) as far as the digest of ref shows it (a lower bound of the full figure)."""
    return digest_err(x, d, 0.0, float(d['max']))


def golden_digests(name):
    """tests/golden/<name>.npz written by tests/golden/make_reference_kernels.py: {'<key>_<field>': array} -> {key: digest}"""
    out = {}
    for k, v in golden(name).items():
        key, field = k.rsplit('_', 1)
        out.setdefault(key, {})[field] = v
    return out


@pytest.fixture(scope='session')
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch.device('cuda:0')
