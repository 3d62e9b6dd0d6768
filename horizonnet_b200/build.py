"""Builds libhorizonnet_b200.so in-tree with nvcc for sm_100a (no torch extension machinery:
the boundary is a plain C ABI loaded with ctypes).  The .so is git-ignored but travels to the GPU
box with the gpurun snapshot.  The digest of the sources is embedded in the binary (hn_build_digest) and the
binding compares it with the checked-out sources, so a stale binary can never be loaded silently; the
`.sha256` stamp beside the .so (untracked, like the .so) only decides whether a rebuild is needed."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'lib', 'libhorizonnet_b200.so')
SOURCES = ['model.cu', 'conv_f32.cu', 'conv_tc.cu', 'tail.cu', 'lstm.cu', 'lstm_cluster.cu', 'panostretch.cu', 'rotate.cu', 'tta.cu', 'layout.cu', 'train_fwd.cu', 'bwd_kernels.cu', 'wgrad_tc.cu', 'train_step.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-cudart', 'static']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), 'include')):
        for name in sorted(os.listdir(root)):
            if name.endswith(('.cu', '.cuh', '.h')):
                h.update(name.encode())
                h.update(open(os.path.join(root, name), 'rb').read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def source_digest():
    """Digest of the CUDA sources, headers and flags; embedded in the .so as hn_build_digest()."""
    return _digest()


def build(force=False, verbose=False):
    """Compile every .cu of the package for sm_100a and link the shared library."""
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    stamp = LIB + '.sha256'
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    objdir = os.path.join(HERE, 'lib', 'obj')
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        extra = ['-DHN_BUILD_DIGEST="%s"' % digest] if src == 'model.cu' else []
        cmd = [nvcc] + NVCC_FLAGS + extra + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f'nvcc failed on {src}')
        objs.append(obj)
    cmd = [nvcc] + NVCC_FLAGS + ['-shared', '-o', LIB] + objs
    subprocess.check_call(cmd)
    open(stamp, 'w').write(digest)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
