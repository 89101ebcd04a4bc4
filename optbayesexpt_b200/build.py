"""Builds optbayesexpt_b200/libobe_b200.so in-tree with nvcc for sm_100a.

    python -m optbayesexpt_b200.build [--force]

nvcc cross-compiles without a GPU.  The two device headers are also embedded as string
literals (csrc/*_src.inc) so that NVRTC can compile user model source against them at run time.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libobe_b200.so')
SOURCES = ['obe_b200.cu', 'obe_device.cuh', 'obe_models.cuh', 'obe_summary.cuh']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-shared', '-Xcompiler', '-fPIC', '-cudart', 'static']


def _embed(header):
    src = open(os.path.join(CSRC, header)).read()
    assert ')OBESRC"' not in src
    # split into chunks: some front ends cap a single string literal at 64 KiB
    chunks, step = [], 12000
    for i in range(0, len(src), step):
        chunks.append('R"OBESRC(' + src[i:i + step] + ')OBESRC"')
    out = os.path.join(CSRC, header.replace('.cuh', '_src.inc'))
    text = '\n'.join(chunks) + '\n'
    if not os.path.exists(out) or open(out).read() != text:
        open(out, 'w').write(text)
    return out


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(HERE, '..', 'include', 'obe_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """``defines`` / ``out``: A/B builds of tuning variants (-DNAME=VALUE ..., written next to the library;
    select one at run time with OBE_B200_LIB=<path>)."""
    if not force and not defines and not needs_build():
        return LIB
    _embed('obe_device.cuh')
    _embed('obe_models.cuh')
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + [f'-D{d}' for d in defines] + \
        ['-o', out or LIB, os.path.join(CSRC, 'obe_b200.cu'), '-ldl']
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out or LIB


if __name__ == '__main__':
    defs = [a[2:] for a in sys.argv[1:] if a.startswith('-D')]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith('--out=')]
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv, defines=defs, out=outs[0] if outs else None))
