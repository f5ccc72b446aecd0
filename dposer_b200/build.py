"""In-tree build of libdposer_b200.so with nvcc for sm_100a (no torch dependency in the library)."""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, 'csrc')
LIBDIR = os.path.join(PKG, 'lib')
LIB = os.path.join(LIBDIR, 'libdposer_b200.so')
SOURCES = ['api.cu', 'score_simt.cu', 'score_tc.cu', 'score_small.cu', 'sampler.cu', 'lbs.cu', 'lbs_bwd.cu', 'lbs_bwd_tc.cu', 'lbs_skin_bwd_tc.cu', 'lbs_tc.cu', 'lbs_fused2.cu', 'lbs_fused3.cu', 'metrics.cu', 'fit.cu', 'fitstep.cu', 'gemm_tc.cu', 'train.cu', 'rk45.cu', 'selfisect.cu', 'procrustes.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _nvcc():
    exe = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(exe):
        raise RuntimeError('nvcc not found: cannot build libdposer_b200.so')
    return exe


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG, '..', 'include', 'dposer_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu into objects (parallel) and link the shared library in-tree."""
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    # DPB_BUILD_DEFINES (timing experiments only): an instrumented copy next to the product library
    defines = ['-D' + d for d in os.environ.get('DPB_BUILD_DEFINES', '').split(',') if d]
    lib = LIB.replace('.so', '_prof.so') if defines else LIB
    objdir = os.path.join(PKG, 'build_prof' if defines else 'build')
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        cmd = [nvcc, *NVCC_FLAGS, *defines, '-c', os.path.join(CSRC, src), '-o', obj]
        if verbose:
            cmd.insert(1, '-Xptxas=-v')
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f'nvcc failed on {src}:\n{out}')
        if verbose and out:
            print(out)
        objs.append(obj)
    cmd = [nvcc, '-shared', '-o', lib, *objs]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        raise RuntimeError(f'link failed:\n{out.stdout}')
    return lib


if __name__ == '__main__':
    print(build(force=True, verbose=True))
