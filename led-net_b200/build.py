"""Build libledb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python led-net_b200/build.py [--force]

Objects are cached per source under csrc/build/; the .so lands next to this file so it
travels with the repo snapshot to the GPU box (it is git-ignored, not gpurun-ignored).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OUT = os.path.join(HERE, 'libledb200.so')
SOURCES = ['engine.cu', 'api.cu', 'packed_conv.cu', 'conv_direct.cu', 'conv_tc.cu', 'ladder_tc.cu', 'dappm.cu', 'stem_tc.cu', 'elementwise.cu', 'tail.cu',
           'metrics.cu', 'ohem.cu', 'train.cu', 'wgrad_tc.cu', 'sesp.cu', 'mfaf.cu', 'getb.cu', 'postprocess.cu', 'seam.cu', 'glue.cu', 'augment.cu', 'png.cu',
           'png_decode.cu', 'jpeg_decode.cu', 'cityscapes.cu', 'visualize.cu']
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
         '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr', '-Xptxas', '-v']


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, 'rb') as f:
            h.update(f.read())
    h.update(' '.join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    bdir = os.path.join(CSRC, 'build')
    os.makedirs(bdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    headers.append(os.path.join(os.path.dirname(HERE), 'include', 'ledb200.h'))
    jobs, objs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(bdir, s + '.o')
        stamp = obj + '.sha'
        dig = _digest([src] + headers)
        objs.append(obj)
        if (not force and os.path.exists(obj) and os.path.exists(stamp)
                and open(stamp).read() == dig):
            continue
        jobs.append((src, obj, stamp, dig))

    def compile_one(job):
        src, obj, stamp, dig = job
        r = subprocess.run([NVCC] + FLAGS + ['-c', src, '-o', obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed for {src}:\n{r.stdout}\n{r.stderr}')
        with open(obj + '.log', 'w') as f:
            f.write(r.stdout + r.stderr)
        with open(stamp, 'w') as f:
            f.write(dig)
        return src

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for done in ex.map(compile_one, jobs):
                if verbose:
                    print('compiled', os.path.basename(done))
    if jobs or not os.path.exists(OUT):
        r = subprocess.run([NVCC, '-shared', '-o', OUT] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a',
                                                                   '-lcudart'],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
