"""Build librelnet_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python relation-networks-for-object-detection_b200/build.py [--force]

One object per .cu (parallel), then one shared library next to this file.  Files whose arithmetic must be
bit-comparable with the CPU oracle are compiled with -fmad=false (see the header comment of each).
"""
import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
INC = os.path.join(os.path.dirname(HERE), 'include')
# measurement variant (tools/fused_trace.py): RELNET_VARIANT=trace builds build_trace/librelnet_b200_trace.so with
# -DRN_FUSED_TRACE next to, never instead of, the product library
VARIANT = os.environ.get('RELNET_VARIANT', '')
OBJ = os.path.join(HERE, 'build' + ('_' + VARIANT if VARIANT else ''))
LIB = os.path.join(OBJ, 'librelnet_b200_%s.so' % VARIANT) if VARIANT else os.path.join(HERE, 'librelnet_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')

COMMON = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
          '-I' + INC, '-I' + CSRC, '--expt-relaxed-constexpr', '-Xptxas', '-v']
NO_FMA = {'rois.cu', 'psroi.cu', 'deform_conv.cu', 'proposal.cu'}


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith('.cu'))


def _stamp():
    h = hashlib.sha1()
    for d in (CSRC, INC):
        for f in sorted(os.listdir(d)):
            with open(os.path.join(d, f), 'rb') as fh:
                h.update(f.encode()); h.update(fh.read())
    with open(__file__, 'rb') as fh:
        h.update(fh.read())
    return h.hexdigest()


def _compile(src):
    obj = os.path.join(OBJ, src[:-3] + '.o')
    cmd = [NVCC] + COMMON + (['-fmad=false'] if src in NO_FMA else []) + (['-DRN_FUSED_TRACE'] if VARIANT == 'trace' else []) + ['-D' + d for d in os.environ.get('RELNET_DEFINES', '').split() if VARIANT] + \
        ['-c', os.path.join(CSRC, src), '-o', obj]
    p = subprocess.run(cmd, capture_output=True, text=True)
    return src, obj, p.returncode, p.stdout + p.stderr


def current():
    """True when the library exists and was built from the present sources.  Reads only: usable on a read-only tree."""
    stamp_file = os.path.join(OBJ, 'stamp')
    return os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == _stamp()


def build(force=False, verbose=False):
    if not force and current():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    stamp_file = os.path.join(OBJ, 'stamp')
    stamp = _stamp()
    objs, logs = [], []
    with cf.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 4)) as ex:
        for src, obj, rc, log in ex.map(_compile, sources()):
            logs.append('== %s\n%s' % (src, log))
            if rc != 0:
                sys.stderr.write('\n'.join(logs))
                raise RuntimeError('nvcc failed on %s' % src)
            objs.append(obj)
    with open(os.path.join(OBJ, 'ptxas.log'), 'w') as f:
        f.write('\n'.join(logs))
    # -gencode at link time as well: the (empty) device-link stub is then sm_100a too, not nvcc's default architecture
    cmd = [NVCC, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs + ['-lcublas', '-Xlinker', '-rpath,/usr/local/cuda/lib64']
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout + p.stderr)
        raise RuntimeError('link failed')
    with open(stamp_file, 'w') as f:
        f.write(stamp)
    if verbose:
        print('\n'.join(logs))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
