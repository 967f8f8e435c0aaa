"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/b200rec.h declares,
the ctypes table covers all of them, and the product path refuses to run without CUDA (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, 'include', 'b200rec.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(b200rec_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    from deeprecommendation_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), 'build first: python -m deeprecommendation_b200.csrc.build'
    h = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(h, n), f'{n} declared in include/b200rec.h but not exported'
    assert set(_lib.SIGNATURES) == set(names), set(_lib.SIGNATURES) ^ set(names)
    lib = _lib.lib()
    header_version = int(re.search(r'#define\s+B200REC_VERSION\s+(\d+)', open(os.path.join(ROOT, 'include', 'b200rec.h')).read()).group(1))
    assert lib.b200rec_version() == header_version == _lib.ABI_VERSION


def test_struct_layouts_match_header_field_order():
    from deeprecommendation_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'b200rec.h')).read()
    for cname, cls in (('b200rec_attention_t', _lib.AttentionDesc), ('b200rec_attention_bwd_t', _lib.AttentionBwdDesc), ('b200rec_spmm_t', _lib.SpmmDesc), ('b200rec_spmm_stream_t', _lib.SpmmStreamDesc), ('b200rec_mlp_t', _lib.MlpDesc)):
        body = re.search(r'typedef struct \{([^}]*)\} ' + cname, src).group(1)
        body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
        fields = []
        for decl in body.split(';'):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(','):
                fields.append(re.sub(r'\[.*\]', '', part.strip().split()[-1].lstrip('*')))
        assert fields == [f[0] for f in cls._fields_], (cname, fields)


def test_workspace_queries_run_without_gpu():
    from deeprecommendation_b200 import _lib
    lib = _lib.lib()
    assert lib.b200rec_scan_workspace(10_000_000) > 0
    assert lib.b200rec_sort_pairs_workspace(1 << 20) >= 2 * 4 * (1 << 20)
    assert lib.b200rec_csr_workspace(1000, 100) > 0
    # argument checks run on the host too: the tensor-core GEMMs refuse a NULL packed_w before any launch
    X, W, Y = 256, 512, 768                                   # never dereferenced
    with pytest.raises(ValueError, match='packed'):
        _lib.check(lib.b200rec_linear_tc(X, 128, 64, 64, W, 64, 64, None, None, 0, Y, 64, _lib.F32, _lib.TC_TF32X3, None, None, 0, None), 'linear_tc')
    with pytest.raises(ValueError, match='packed'):
        _lib.check(lib.b200rec_linear_tc_splitk(X, 128, 64, 64, W, 64, 64, None, None, 0, Y, 64, _lib.F32, _lib.TC_TF32X3, None, None, 0, None),
                   'linear_tc_splitk')
    prob = _lib.LinearProblem(X=X, M=128, ldx=64, W=W, N=64, ldw=64, packed_w=None, Y=Y, ldy=64, y_dtype=_lib.F32)
    with pytest.raises(ValueError, match='packed'):
        _lib.check(lib.b200rec_linear_tc_batch(ctypes.byref(prob), 1, 64, _lib.TC_TF32X3, None), 'linear_tc_batch')


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU behaviour')
def test_no_cpu_fallback():
    from deeprecommendation_b200.neural_collaborative_filtering.models import BasicNCF
    m = BasicNCF(8, 8, item_emb=4, user_emb=4, mlp_dense_layers=[8]).eval()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m(torch.zeros(2, 8), torch.zeros(2, 8))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, 'deeprecommendation_b200')
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                txt = open(os.path.join(d, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', txt, flags=re.M), f'{f} imports the oracle'


def test_header_is_plain_c():
    """The boundary is a C ABI: include/b200rec.h must compile as C99 with no C++ / CUDA / torch types in any signature."""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('no gcc')
    header = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'b200rec.h')
    r = subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-fsyntax-only', '-x', 'c', header], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
