"""In-tree nvcc build of libmpe_b200.so (sm_100a only).

    python -m multiagent_rl_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the
repo snapshot.  The fp64 env kernels are built with -fmad=false (validation build: every product and
sum rounds like the float64 numpy reference).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(HERE, 'csrc', 'build')
LIB = os.path.join(HERE, 'libmpe_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden']

UNITS = [
    ('env_kernels_f32.cu', []),
    ('env_kernels_f64.cu', ['-fmad=false']),
    ('actor_kernels.cu', []),
    ('tc_kernels.cu', []),
    ('replay_kernels.cu', []),
    ('critic_kernels.cu', []),
    ('critic_grad_kernels.cu', []),
    ('actor_grad_kernels.cu', []),
    ('grad_reduce.cu', []),
    ('pack_kernels.cu', []),
    ('cabi.cu', ['-Xcompiler', '-fvisibility=default']),
]


def _sources():
    files = sorted(f for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh', '.h')))
    files = [os.path.join(CSRC, f) for f in files]
    files.append(os.path.join(os.path.dirname(HERE), 'include', 'mpe_b200.h'))
    files.append(os.path.abspath(__file__))
    return files


def source_hash():
    h = hashlib.sha256()
    for f in _sources():
        with open(f, 'rb') as fp:
            h.update(fp.read())
    return h.hexdigest()


def up_to_date():
    stamp = LIB + '.hash'
    return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == source_hash()


def _compile(unit):
    src, extra = unit
    obj = os.path.join(OBJ, src.replace('.cu', '.o'))
    cmd = [NVCC] + ARCH + COMMON + extra + ['-c', os.path.join(CSRC, src), '-o', obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('nvcc failed for %s:\n%s\n%s' % (src, ' '.join(cmd), r.stderr[-4000:]))
    return obj


def build(force=False, verbose=True):
    if not force and up_to_date():
        return LIB
    if not os.path.exists(NVCC):
        raise RuntimeError('nvcc not found at %s; libmpe_b200.so cannot be built' % NVCC)
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(_compile, UNITS))
    cmd = [NVCC] + ARCH + ['-shared', '-o', LIB] + objs + ['-lcudart_static', '-ldl', '-lrt', '-lpthread']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n%s' % r.stderr[-4000:])
    with open(LIB + '.hash', 'w') as fp:
        fp.write(source_hash())
    if verbose:
        print('built', LIB)
    return LIB


def build_variant(name, defines):
    """A/B or instrumented build next to the product library (tools/; load it with MPE_B200_LIB=...):
    tmp_ab/libmpe_b200_<name>.so compiled with the given -D defines."""
    out_dir = os.path.join(os.path.dirname(HERE), 'tmp_ab')
    obj_dir = os.path.join(out_dir, name)
    os.makedirs(obj_dir, exist_ok=True)

    def one(unit):
        src, extra = unit
        obj = os.path.join(obj_dir, src.replace('.cu', '.o'))
        cmd = [NVCC] + ARCH + COMMON + extra + ['-D' + d for d in defines] + ['-c', os.path.join(CSRC, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (src, r.stderr[-4000:]))
        return obj

    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(one, UNITS))
    lib = os.path.join(out_dir, 'libmpe_b200_%s.so' % name)
    r = subprocess.run([NVCC] + ARCH + ['-shared', '-o', lib] + objs + ['-lcudart_static', '-ldl', '-lrt', '-lpthread'],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n%s' % r.stderr[-4000:])
    print('built', lib)
    return lib


if __name__ == '__main__':
    if '--variant' in sys.argv:  # python -m multiagent_rl_b200.build --variant phases MPE_TC_PHASES
        i = sys.argv.index('--variant')
        build_variant(sys.argv[i + 1], sys.argv[i + 2:])
    else:
        build(force='--force' in sys.argv)
