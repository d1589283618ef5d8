"""In-tree build of the CUDA library (``liblatentaugment_b200.so``) with nvcc for sm_100a.

``python -m latentaugment_b200._build`` or ``__graft_entry__.build()``.  nvcc
cross-compiles without a GPU.  The library links the static CUDA runtime and exposes only
the C ABI of ``include/latentaugment_b200.h``.

Staleness is decided by CONTENT hashes (source + headers + flags), not mtimes: the hashes of what
each object / the library was built from are stored next to them, so a checkout that changed a
source rebuilds exactly the affected objects and a snapshot copied to another machine (mtimes
shuffled) rebuilds nothing.
"""
import hashlib
import json
import os
import re
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, 'csrc')
LIB = os.path.join(PKG, 'liblatentaugment_b200.so')
STAMP = LIB + '.srchash'
SOURCES = ['tapgemm.cu', 'kernels.cu', 'distance.cu', 'engine.cu', 'disc.cu', 'filtered_lrelu.cu', 'lpips.cu', 'detector.cu']
HEADERS = ['act.cuh', 'common.cuh', 'tapgemm.cuh', 'kernels.cuh', 'sm100.cuh', 'plan.cuh', 'disc.cuh', 'lpips.cuh', 'vgg.cuh',
           os.path.join(ROOT, 'include', 'latentaugment_b200.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _sha(paths, extra=''):
    h = hashlib.sha256(extra.encode())
    for p in paths:
        with open(p, 'rb') as f:
            h.update(f.read())
    return h.hexdigest()


def _header_paths():
    return [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]


def _deps(path, seen=None):
    """The file plus every project header it includes with quotes, transitively."""
    seen = seen if seen is not None else []
    path = os.path.normpath(path)
    if path in seen or not os.path.exists(path):
        return seen
    seen.append(path)
    for m in re.finditer(r'^\s*#\s*include\s+"([^"]+)"', open(path).read(), re.M):
        _deps(os.path.join(os.path.dirname(path), m.group(1)), seen)
    return seen


def source_hashes():
    """{source: hash of (that source, the headers it includes, the flags)}."""
    known = set(os.path.normpath(h) for h in _header_paths())
    out = {}
    for s in SOURCES:
        deps = _deps(os.path.join(CSRC, s))
        missing = [d for d in deps[1:] if d not in known]
        assert not missing, f'{s} includes headers that HEADERS does not list: {missing}'
        out[s] = _sha(deps, ' '.join(NVCC_FLAGS))
    return out


def _stored():
    try:
        return json.load(open(STAMP))
    except (OSError, ValueError):
        return {}


def stale():
    return not os.path.exists(LIB) or _stored() != source_hashes()


def build(force=False, verbose=False):
    want = source_hashes()
    have = {} if force else _stored()
    if not force and os.path.exists(LIB) and have == want:
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(PKG, 'build'), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(PKG, 'build', src.replace('.cu', '.o'))
        objs.append(obj)
        if not force and os.path.exists(obj) and have.get(src) == want[src]:
            continue
        cmd = [_nvcc()] + NVCC_FLAGS + ['-c', os.path.join(CSRC, src), '-o', obj]
        if verbose:
            print(' '.join(cmd), file=sys.stderr)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = []
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed.append(f'nvcc failed on {src}:\n{out}')
        elif verbose and out.strip():
            print(out, file=sys.stderr)
    if failed:
        if os.path.exists(STAMP):
            os.remove(STAMP)
        raise RuntimeError('\n'.join(failed))
    cmd = [_nvcc(), '-shared'] + NVCC_FLAGS[:2] + ['-o', LIB] + objs      # (-gencode here too: no default-arch stub cubin in the library)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'link failed:\n{r.stdout}')
    json.dump(want, open(STAMP, 'w'))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
