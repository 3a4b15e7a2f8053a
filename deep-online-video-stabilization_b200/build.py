"""Builds libmgw_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python deep-online-video-stabilization_b200/build.py [--force] [--verbose]

-fmad=false: the reference's fp32 rounding order is part of the contract (parity is bit-exact on the per-pixel
stage), so nvcc must never contract a*b+c on its own; every fused multiply-add in csrc/ is an explicit fmaf.
cudart is linked statically and the driver API is reached through cudaGetDriverEntryPoint, so the library
loads (and exports its symbols) on a box without libcuda.so.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
SO = os.path.join(HERE, os.environ.get('MGW_SO_NAME', 'libmgw_b200.so'))       # MGW_SO_NAME / MGW_EXTRA_FLAGS: A/B builds for tuning
SOURCES = ['mgw_capi.cu', 'mgw_solve.cu', 'mgw_warp_generic.cu', 'mgw_warp_tma.cu', 'mgw_warp_pipe.cu', 'mgw_interp.cu', 'mgw_loss.cu', 'mgw_loss_tile.cu', 'mgw_pass.cu', 'mgw_deploy.cu', 'mgw_stream.cu', 'mgw_crop.cu', 'mgw_vertex_loss.cu']
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-fmad=false',
         '--expt-relaxed-constexpr', '-Xcompiler', '-fPIC,-O2,-fvisibility=hidden', '-cudart', 'static']


def _deps():
    d = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    d.append(os.path.join(os.path.dirname(HERE), 'include', 'mgw.h'))
    d.append(os.path.abspath(__file__))
    return d


def build(force=False, verbose=False):
    if not force and os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(p) for p in _deps()):
        return SO
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objs = []
    bdir = os.path.join(HERE, 'build', os.path.basename(SO))
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(bdir, src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [nvcc] + FLAGS + os.environ.get('MGW_EXTRA_FLAGS', '').split() + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write('--- %s\n%s\n' % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed')
    subprocess.check_call([nvcc, '-shared', '-cudart', 'static', '-o', SO] + objs)
    return SO


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
