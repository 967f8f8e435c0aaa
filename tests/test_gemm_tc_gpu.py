"""K1a on tcgen05 (csrc/gemm_tc.cu): hand-written tensor-core GEMM vs an fp64 reference.
TF32x3 mode must stay inside the fp32 parity tolerance (max-norm rel <= 1e-5); bf16 mode inside 1e-2."""
import pytest
import torch

from tests._golden import maxnorm_rel

pytestmark = pytest.mark.gpu
SHAPES = [(128, 64, 128), (128, 32, 128), (300, 2094, 256), (9447, 2094, 256), (1000, 128, 128), (129, 70, 17), (4096, 2093, 130),
          (50000, 128, 128)]


def _case(M, K, N, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    s = torch.rand(M, generator=g) + 0.5
    return x, w, b, s


@pytest.mark.parametrize('M,K,N', SHAPES)
def test_linear_tc_tf32x3_fp32_parity(M, K, N):
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + K)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    y = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='tf32x3!')
    assert maxnorm_rel(y, ref) < 1e-5
    # epilogue: row scale + relu, strided output
    out = torch.full((M, N + 8), 3.0, device='cuda')
    ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), s.cuda(), True, out=out[:, 4:4 + N], engine='tf32x3!')
    ref2 = (ref * s.double()[:, None]).relu()
    assert maxnorm_rel(out[:, 4:4 + N], ref2) < 1e-5
    assert torch.all(out[:, :4] == 3.0) and torch.all(out[:, 4 + N:] == 3.0)


@pytest.mark.parametrize('M,K,N', [(512, 2094, 256), (512, 2094, 128), (128, 2094, 128), (1000, 2093, 132), (257, 1024, 64), (2000, 4096, 256),
                                   (256, 4731, 2094), (512, 2094, 130), (300, 1000, 17), (128, 640, 1)])
def test_linear_tc_splitk_fp32_parity(M, K, N):
    """short-M, long-K shapes (a batch of pairs against the F-wide profiles) take the split-K tensor-core route of `linear_raw`:
    same tolerance, bit-reproducible (the slabs are added in split order), epilogue applied after the reduction"""
    from deeprecommendation_b200 import _lib as L
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + K + 7)
    assert L.lib().b200rec_linear_tc_splitk_workspace(M, N, K, L.TC_TF32X3) > 0
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    timer = ops.OpTimer()
    ops.set_timer(timer)
    try:
        y = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='tf32x3')
    finally:
        ops.set_timer(None)
    torch.cuda.synchronize()
    assert any(name == 'linear_tc_splitk' for name, _ in timer.summary())
    assert maxnorm_rel(y, ref) < 1e-5
    assert torch.equal(y, ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='tf32x3'))
    out = torch.full((M, N + 8), 3.0, device='cuda')
    ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), s.cuda(), True, out=out[:, 4:4 + N], engine='tf32x3')
    assert maxnorm_rel(out[:, 4:4 + N], (ref * s.double()[:, None]).relu()) < 1e-5
    assert torch.all(out[:, :4] == 3.0) and torch.all(out[:, 4 + N:] == 3.0)
    yb = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), out_dtype=torch.bfloat16, engine='tf32x3')
    assert yb.dtype == torch.bfloat16 and maxnorm_rel(yb.float(), ref) < 1e-2


@pytest.mark.parametrize('M,K,N', SHAPES[:5])
def test_linear_tc_bf16(M, K, N):
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + K + 1)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    y = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='bf16!')
    assert maxnorm_rel(y, ref) < 1e-2
    yb = ops.linear_raw(x.cuda(), w.cuda(), None, out_dtype=torch.bfloat16, engine='bf16!')
    assert yb.dtype == torch.bfloat16 and maxnorm_rel(yb.float(), x.double() @ w.double().T) < 1e-2


def test_linear_tc_real_profiles():
    """the reference's own input statistics: sparse binary block + dense [0,1) block, F = 2094 (8-byte aligned rows)"""
    from deeprecommendation_b200 import ops, synth
    x = torch.from_numpy(synth.item_profiles(3000, seed=3))
    sd = synth.to_torch(synth.attention_ncf_weights(2094, seed=2))
    w = torch.cat((sd['ItemEmbeddings.0.weight'], sd['UserEmbeddings.0.weight']))
    b = torch.cat((sd['ItemEmbeddings.0.bias'], sd['UserEmbeddings.0.bias']))
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    y = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='tf32x3!')
    simt = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='simt')
    assert maxnorm_rel(y, ref) < 1e-5 and maxnorm_rel(simt, ref) < 1e-5


@pytest.mark.parametrize('M,K,N', [(5000, 128, 128), (130, 64, 64), (100_000, 128, 128), (777, 96, 100), (20_000, 32, 8), (1, 128, 128),
                                   (162_541, 128, 128)])
def test_linear_shortk_persistent_fp32_parity(M, K, N):
    """K1c (csrc/node_gemm.cu): persistent short-K tcgen05 GEMM of the per-node transforms, 3xTF32 -> fp32 tolerance"""
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + K + 7)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    y = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='shortk!')
    assert y.shape == (M, N) and maxnorm_rel(y, ref) < 1e-5
    # row scale + relu, strided input (column slice of a wider buffer) and strided output
    xw = torch.zeros(M, K + 32, device='cuda')
    xw[:, 16:16 + K] = x.cuda()
    out = torch.full((M, N + 8), 3.0, device='cuda')
    ops.linear_raw(xw[:, 16:16 + K], w.cuda(), None, s.cuda(), True, out=out[:, 4:4 + N], engine='shortk!')
    ref2 = (torch.nn.functional.linear(x.double(), w.double()) * s.double()[:, None]).relu()
    assert maxnorm_rel(out[:, 4:4 + N], ref2) < 1e-5
    assert torch.all(out[:, :4] == 3.0) and torch.all(out[:, 4 + N:] == 3.0)
    # the automatic dispatch of the default tensor-core engine picks it for large M and gives the same bits
    if M >= ops.SHORTK_MIN_ROWS:
        y2 = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), engine='tf32x3')
        assert torch.equal(y, y2)


@pytest.mark.parametrize('M,K,N', [(5000, 128, 128), (777, 96, 100), (20_000, 32, 8), (1, 128, 128)])
def test_linear_shortk_bf16_output(M, K, N):
    """K1c with a bf16 epilogue (GraphNCF.message_dtype = 'bf16'): the fp32 result rounded once, bit-identical to rounding the
    fp32-output run; strided output leaves its neighbours alone"""
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + K + 11)
    y32 = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), s.cuda(), engine='shortk!')
    y16 = ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), s.cuda(), out_dtype=torch.bfloat16, engine='shortk!')
    assert y16.dtype == torch.bfloat16 and torch.equal(y16, y32.bfloat16())
    out = torch.full((M, N + 12), 3.0, device='cuda', dtype=torch.bfloat16)
    ops.linear_raw(x.cuda(), w.cuda(), b.cuda(), s.cuda(), out=out[:, 6:6 + N], engine='shortk!')       # rows only 4-byte aligned
    assert torch.equal(out[:, 6:6 + N], y16) and torch.all(out[:, :6] == 3.0) and torch.all(out[:, 6 + N:] == 3.0)


@pytest.mark.parametrize('Ma,Mb,K,Na,Nb', [(512, 512, 2094, 128, 128), (300, 129, 2094, 256, 64), (512, 512, 700, 128, 128), (100, 512, 2094, 128, 128)])
def test_linear_pair_batched_splitk(Ma, Mb, K, Na, Nb):
    """BasicNCF's two projections in one split-K launch (b200rec_linear_tc_splitk_batch): fp32 parity for both outputs; shapes the batch
    does not cover (M below the split-K window) fall through to two single launches with the same results"""
    from deeprecommendation_b200 import ops
    xa, wa, ba, _ = _case(Ma, K, Na, 3)
    xb, wb, bb, _ = _case(Mb, K, Nb, 4)
    prev = ops.set_gemm_engine('tf32x3')
    try:
        ya, yb = ops.linear_pair(xa.cuda(), wa.cuda(), ba.cuda(), xb.cuda(), wb.cuda(), bb.cuda())
    finally:
        ops.set_gemm_engine(prev)
    assert maxnorm_rel(ya, torch.nn.functional.linear(xa.double(), wa.double(), ba.double())) < 1e-5
    assert maxnorm_rel(yb, torch.nn.functional.linear(xb.double(), wb.double(), bb.double())) < 1e-5


@pytest.mark.parametrize('M,K,N', [(9461, 2094, 256), (2500, 2094, 256), (4096, 512, 384 + 128), (3000, 1000, 130), (2049, 2094, 200)])
def test_linear_tc_wide_tiles_fp32_parity_vs_128_tiles(M, K, N):
    """128 x 256 tiles + split-K (b200rec_linear_tc_wide): the default route of large-M GEMMs with 128 < N.  Same fp32 tolerance as the
    128 x 128 form, deterministic, agrees with it to fp32 rounding; row_index gather, bias / row scale / ReLU after the slab reduction."""
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + N)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    xd, wd, bd, sd = x.cuda(), w.cuda(), b.cuda(), s.cuda()
    y = ops.linear_raw(xd, wd, bd, engine='tf32x3!')
    assert maxnorm_rel(y, ref) < 1e-5
    assert torch.equal(y, ops.linear_raw(xd, wd, bd, engine='tf32x3!'))
    y128 = ops.linear_tc_batch([(xd, wd, bd, None)], engine='tf32x3')[0]          # the 128 x 128 tiles
    assert maxnorm_rel(y, y128) < 2e-6
    out = torch.full((M, N + 8), 3.0, device='cuda')
    ops.linear_raw(xd, wd, bd, sd, True, out=out[:, 4:4 + N], engine='tf32x3!')
    assert maxnorm_rel(out[:, 4:4 + N], (ref * s.double()[:, None]).relu()) < 1e-5
    assert torch.all(out[:, :4] == 3.0) and torch.all(out[:, 4 + N:] == 3.0)
    idx = torch.randint(0, M, (2300,), generator=torch.Generator().manual_seed(1)).cuda()
    yg = ops.linear_raw(xd, wd, bd, row_index=idx, engine='tf32x3!')
    assert maxnorm_rel(yg, ref[idx.cpu()]) < 1e-5


@pytest.mark.parametrize('M,K,N', [(9461, 2094, 256), (2500, 2094, 256), (4096, 512, 384 + 128), (3000, 1000, 130), (2049, 2093, 200), (2100, 2096, 256)])
def test_linear_tc_wide_bf16x3_split(M, K, N):
    """The opt-in bf16 hi/lo engine of the wide form (B200REC_TC_BF16X3): the three products of the 3xTF32 scheme on 16-bit-mantissa operands.
    Budget 1e-5 of the largest output (measured ~4e-6 at K = 2094); deterministic; 64-bit, scalar (odd K) and 128-bit producer loads."""
    from deeprecommendation_b200 import ops
    x, w, b, s = _case(M, K, N, M + N + 1)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double())
    xd, wd, bd, sd = x.cuda(), w.cuda(), b.cuda(), s.cuda()
    y = ops.linear_raw(xd, wd, bd, engine='bf16x3!')
    err = maxnorm_rel(y, ref)
    assert err < 1e-5, err
    assert torch.equal(y, ops.linear_raw(xd, wd, bd, engine='bf16x3!'))
    y3 = ops.linear_raw(xd, wd, bd, engine='tf32x3!')
    assert not torch.equal(y, y3)                                   # it really is the other engine
    out = torch.full((M, N + 8), 3.0, device='cuda')
    ops.linear_raw(xd, wd, bd, sd, True, out=out[:, 4:4 + N], engine='bf16x3!')
    assert maxnorm_rel(out[:, 4:4 + N], (ref * s.double()[:, None]).relu()) < 1e-5
    assert torch.all(out[:, :4] == 3.0) and torch.all(out[:, 4 + N:] == 3.0)
    idx = torch.randint(0, M, (2300,), generator=torch.Generator().manual_seed(1)).cuda()
    assert maxnorm_rel(ops.linear_raw(xd, wd, bd, row_index=idx, engine='bf16x3!'), ref[idx.cpu()]) < 1e-5
    # binary (multi-hot) rows are exact in bf16: only W's split error remains
    xb = (torch.rand(M, K, generator=torch.Generator().manual_seed(5)) < 0.02).float()
    eb = maxnorm_rel(ops.linear_raw(xb.cuda(), wd, bd, engine='bf16x3!'), torch.nn.functional.linear(xb.double(), w.double(), b.double()))
    assert eb < 5e-6, eb
