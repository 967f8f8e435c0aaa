"""Build libb200rec.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m deeprecommendation_b200.csrc.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(os.path.dirname(HERE), 'libb200rec.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
SOURCES = ['api.cu', 'gemm_f32.cu', 'gemm_tc.cu', 'mlp_tower.cu', 'attention_pool.cu', 'attention_pool_bwd.cu', 'spmm.cu', 'graph_build.cu', 'topk.cu', 'allpairs.cu', 'node_gemm.cu', 'peer.cu', 'gather_sum.cu', 'spmm_stream.cu', 'attention_pool_drop.cu', 'collate.cu', 'neg_sample.cu', 'attention_recommend.cu', 'attention_explain.cu']
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
         '--expt-relaxed-constexpr', '-I', os.path.join(ROOT, 'include')]


def _deps():
    d = [os.path.join(HERE, s) for s in SOURCES]
    d += [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith('.cuh')]
    d.append(os.path.join(ROOT, 'include', 'b200rec.h'))
    return d


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    extra = ['-Xptxas', '-v'] if verbose else []

    def compile_one(src):
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        srcp = os.path.join(HERE, src)
        included = [os.path.join(HERE, 'attention_pool.cu')] if src == 'attention_pool_drop.cu' else []     # (that unit #includes the other one)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(
                os.path.getmtime(p) for p in [srcp] + included + [d for d in _deps() if not d.endswith('.cu')]):
            return obj, ''
        r = subprocess.run([NVCC] + FLAGS + extra + ['-c', srcp, '-o', obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed on {src}:\n{r.stdout}\n{r.stderr}')
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        results = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, log in results:
            if log:
                print(log)
    objs = [o for o, _ in results]
    r = subprocess.run([NVCC, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart'],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
