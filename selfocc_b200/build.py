"""Build libselfocc_b200.so in-tree with nvcc for sm_100a (no torch types, plain C ABI)."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, 'csrc')
LIB_DIR = os.path.join(PKG, 'lib')
LIB = os.path.join(LIB_DIR, 'libselfocc_b200.so')
SOURCES = ['abi.cu', 'render.cu', 'render_fast.cu', 'field_hess.cu', 'metric.cu', 'occupancy.cu', 'render_train.cu', 'decode.cu', 'msda.cu', 'gemm.cu', 'norm.cu']
# approx-unit math (ex2/rcp/rsq) without the denormal range-scaling wrappers: ~20 instructions per render sample
PER_SOURCE_FLAGS = {'render.cu': ['-ftz=true'], 'render_fast.cu': ['-ftz=true'], 'render_train.cu': ['-ftz=true'],
                    'occupancy.cu': ['-ftz=true'],   # same field-query arithmetic as so_field_query (render.cu)
                    'msda.cu': ['-ftz=true'], 'decode.cu': ['-ftz=true']}
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '--expt-relaxed-constexpr', '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG, '..', 'include', 'selfocc_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, out=None, defines=()):
    """out/defines: build an experimental variant (e.g. out='libexp.so', defines=['-DSO_RENDER_UNROLL=4']) next to the
    default library; select it at run time with SELFOCC_B200_LIB=<path>."""
    if out is None and not force and not needs_build():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    tag = '' if out is None else '.' + os.path.splitext(os.path.basename(out))[0]
    objs = []
    procs = []
    srcs = list(SOURCES)
    missing = [s for s in srcs if not os.path.exists(os.path.join(CSRC, s))]
    if missing:
        raise RuntimeError('CUDA sources missing from %s: %s' % (CSRC, missing))
    for s in srcs:
        o = os.path.join(LIB_DIR, s.replace('.cu', tag + '.o'))
        objs.append(o)
        cmd = [_nvcc()] + NVCC_FLAGS + PER_SOURCE_FLAGS.get(s, []) + list(defines) + ['-c', os.path.join(CSRC, s), '-o', o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for s, p in procs:
        text, _ = p.communicate()
        log.append('== %s\n%s' % (s, text))
        if p.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (s, text))
    with open(os.path.join(LIB_DIR, 'build%s.log' % tag), 'w') as f:
        f.write('\n'.join(log))
    if verbose:
        print('\n'.join(log))
    target = LIB if out is None else os.path.join(LIB_DIR, os.path.basename(out))
    cmd = [_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', target] + objs + ['-lcudart']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stdout)
    return target


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
