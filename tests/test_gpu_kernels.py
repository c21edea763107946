"""-m gpu: kernel-level checks of the C-ABI GEMMs against torch fp32 / fp64 matmul on the same inputs.

spv_gemm (fp32 SIMT): relative error <= 1e-5.  spv_tc_gemm (bf16 tcgen05): inputs are rounded to bf16 on both sides,
products accumulate in fp32, so the comparison against torch on the SAME bf16-rounded inputs is <= 1e-4 relative."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("ta,tb", [(0, 1), (0, 0), (1, 0)])
@pytest.mark.parametrize("M,N,K", [(70, 130, 45), (512, 256, 1000), (33, 7, 300)])
def test_simt_gemm(ta, tb, M, N, K):
    from spvipes_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(1)
    A = torch.randn((K, M) if ta else (M, K), generator=g, device="cuda")
    B = torch.randn((N, K) if tb else (K, N), generator=g, device="cuda")
    bias = torch.randn(N, generator=g, device="cuda")
    C = torch.empty(M, N, device="cuda")
    ws = torch.empty(4 * M * N, device="cuda")
    for splits in (1, 4):
        L.check(lib.spv_gemm(0, ta, 0, tb, A.data_ptr(), A.stride(0), None, B.data_ptr(), B.stride(0), None, C.data_ptr(), N, M, N,
                             K, 1, 0, 0, 0, bias.data_ptr(), 0, 1, 0, splits, ws.data_ptr(), _stream()), "spv_gemm")
        torch.cuda.synchronize()
        want = torch.relu((A.t() if ta else A).double() @ (B.t() if tb else B).double() + bias.double())
        err = float((C.double() - want).abs().max() / want.abs().max())
        assert err < 1e-5, (splits, err)


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (1, 1), (0, 1), (1, 0)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (512, 256, 5000), (200, 291, 512), (5000, 40, 512), (96, 64, 136)])
def test_tc_gemm(a_mn, b_mn, M, N, K):
    from spvipes_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(2)
    r8 = lambda x: (x + 7) // 8 * 8
    A = torch.zeros((K, r8(M)) if a_mn else (M, r8(K)), device="cuda", dtype=torch.bfloat16)
    B = torch.zeros((K, r8(N)) if b_mn else (N, r8(K)), device="cuda", dtype=torch.bfloat16)
    if a_mn:
        A[:, :M] = torch.randn(K, M, generator=g, device="cuda").bfloat16()
    else:
        A[:, :K] = torch.randn(M, K, generator=g, device="cuda").bfloat16()
    if b_mn:
        B[:, :N] = torch.randn(K, N, generator=g, device="cuda").bfloat16()
    else:
        B[:, :K] = torch.randn(N, K, generator=g, device="cuda").bfloat16()
    Af = (A[:, :M].t() if a_mn else A[:, :K]).double()
    Bf = (B[:, :N].t() if b_mn else B[:, :K]).double()
    bias = torch.randn(N, generator=g, device="cuda")
    want = Af @ Bf.t() + bias.double()
    ws = torch.empty(8 * M * N, device="cuda")
    for splits in (1, 3):
        C = torch.full((M, N), float("nan"), device="cuda")
        L.check(lib.spv_tc_gemm(a_mn, b_mn, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), C.data_ptr(), N, M, N, K,
                                bias.data_ptr(), 0, 0, splits, ws.data_ptr(), _stream()), "spv_tc_gemm")
        torch.cuda.synchronize()
        err = float((C.double() - want).abs().max() / want.abs().max())
        assert err < 1e-4, (splits, err)


@pytest.mark.parametrize("fmt", [0, 3])
@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (1, 1), (0, 1)])
def test_tc_gemm_operand_formats(fmt, a_mn, b_mn):
    """spv_tc_gemm_ex: bf16 or fp16 operands (both the same: a mixed pair is an illegal instruction on sm_100), alpha scaling"""
    from spvipes_b200 import _lib as L
    lib = L.load()
    M, N, K = 304, 200, 520  # MN-major operands: the leading dimension must be a multiple of 8 elements (TMA pitch)
    g = torch.Generator(device="cuda").manual_seed(6)
    ta, tb = (torch.float16 if fmt & 1 else torch.bfloat16), (torch.float16 if fmt & 2 else torch.bfloat16)
    A = torch.randn((K, M) if a_mn else (M, K), generator=g, device="cuda").to(ta).contiguous()
    B = torch.randn((K, N) if b_mn else (N, K), generator=g, device="cuda").to(tb).contiguous()
    want = 0.5 * ((A.t() if a_mn else A).double() @ (B if b_mn else B.t()).double())
    ws = torch.empty(4 * M * N, device="cuda")
    assert lib.spv_tc_gemm_ex(1, 1.0, a_mn, b_mn, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), ws.data_ptr(), N, M, N, K, None, 0,
                              0, 1, None, _stream()) == -1
    for splits in (1, 3):
        C = torch.full((M, N), float("nan"), device="cuda")
        L.check(lib.spv_tc_gemm_ex(fmt, 0.5, a_mn, b_mn, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), C.data_ptr(), N, M, N, K,
                                   None, 0, 0, splits, ws.data_ptr(), _stream()), "spv_tc_gemm_ex")
        torch.cuda.synchronize()
        err = float((C.double() - want).abs().max() / want.abs().max())
        assert err < 1e-4, (fmt, splits, err)


@pytest.mark.parametrize("a_mn,b_mn,M,N,K", [(0, 0, 512, 256, 5000), (1, 1, 256, 5000, 512), (0, 0, 100, 40, 333)])
def test_tc_gemm_split_is_fp32_grade(a_mn, b_mn, M, N, K):
    """spv_tc_gemm_split (hi.hi + hi.lo + lo.hi on bf16 pairs) against float64 on fp32 operands: ~2^-16 per operand, where the
    plain bf16 GEMM of the same operands is at 2^-9.  Shapes of the encoder fc1 forward / weight gradient at C2."""
    from spvipes_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(4)
    r8 = lambda x: (x + 7) // 8 * 8
    Af = torch.rand(M, K, generator=g, device="cuda") * 3          # like log1p(counts): non-negative, no cancellation help
    Bf = (torch.rand(N, K, generator=g, device="cuda") * 2 - 1) * 0.02
    def planes(X, mn):
        Xs = X.t().contiguous() if mn else X
        hi = torch.zeros(Xs.shape[0], r8(Xs.shape[1]), device="cuda", dtype=torch.bfloat16)
        lo = torch.zeros_like(hi)
        L.check(lib.spv_to_bf16_split(Xs.data_ptr(), Xs.stride(0), hi.data_ptr(), lo.data_ptr(), hi.stride(0), Xs.shape[0], Xs.shape[1],
                                      _stream()), "spv_to_bf16_split")
        return hi, lo
    Ah, Al = planes(Af, a_mn)
    Bh, Bl = planes(Bf, b_mn)
    want = Af.double() @ Bf.double().t()
    ws = torch.empty(8 * M * N, device="cuda")
    for splits in (1, 4):
        C = torch.full((M, N), float("nan"), device="cuda")
        L.check(lib.spv_tc_gemm_split(a_mn, b_mn, Ah.data_ptr(), Al.data_ptr(), Ah.stride(0), Bh.data_ptr(), Bl.data_ptr(), Bh.stride(0),
                                      C.data_ptr(), N, M, N, K, None, 0, 0, splits, ws.data_ptr(), _stream()), "spv_tc_gemm_split")
        torch.cuda.synchronize()
        err = float((C.double() - want).abs().max() / want.abs().max())
        assert err < 5e-5, (splits, err)
    C1 = torch.empty(M, N, device="cuda")
    L.check(lib.spv_tc_gemm(a_mn, b_mn, Ah.data_ptr(), Ah.stride(0), Bh.data_ptr(), Bh.stride(0), C1.data_ptr(), N, M, N, K, None, 0, 0, 1,
                            None, _stream()), "spv_tc_gemm")
    torch.cuda.synchronize()
    assert float((C1.double() - want).abs().max() / want.abs().max()) > 10 * err  # the plain bf16 product is far coarser


@pytest.mark.parametrize("tb", [1, 0])
@pytest.mark.parametrize("M,N,K,batch", [(512, 128, 128, 2), (512, 50, 128, 1), (512, 256, 35, 1), (300, 35, 256, 1), (77, 20, 9, 1)])
def test_smallk_gemm(tb, M, N, K, batch):
    """whole-K variant behind spv_gemm (K <= 256, no split, A not transposed): bias, ReLU, accumulate, batch, odd pitches"""
    from spvipes_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(3)
    lda, ldc = K * batch + 3, N * batch + 1  # batches side by side in the columns, unaligned pitches (scalar staging path)
    A = torch.randn(M, lda, generator=g, device="cuda")
    Bm = torch.randn(batch, N, K, generator=g, device="cuda") if tb else torch.randn(batch, K, N, generator=g, device="cuda")
    bias = torch.randn(batch, N, generator=g, device="cuda")
    C0 = torch.randn(M, ldc, generator=g, device="cuda")
    for relu, acc in ((1, 0), (0, 1)):
        C = C0.clone()
        L.check(lib.spv_gemm(0, 0, 0, tb, A.data_ptr(), lda, None, Bm.data_ptr(), Bm.stride(1), None, C.data_ptr(), ldc, M, N, K,
                             batch, K, Bm.stride(0), N, bias.data_ptr(), N, relu, acc, 1, None, _stream()), "spv_gemm")
        torch.cuda.synchronize()
        for b in range(batch):
            a = A[:, b * K:(b + 1) * K].double()
            w = Bm[b].double()
            want = a @ (w.t() if tb else w) + bias[b].double()
            if relu:
                want = torch.relu(want)
            if acc:
                want = want + C0[:, b * N:(b + 1) * N].double()
            got = C[:, b * N:(b + 1) * N].double()
            err = float((got - want).abs().max() / want.abs().max())
            assert err < 1e-5, (relu, acc, b, err)
        assert torch.equal(C[:, batch * N:], C0[:, batch * N:])  # padding column untouched


def test_adam_ranges_and_staging():
    """spv_adam on sub-ranges with bf16 staging == one launch over the whole vector == torch.optim.Adam semantics"""
    from spvipes_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(5)
    n, rows, cols, off = 4096 + 4 * 37, 31, 37, 1024
    p0 = torch.randn(n, generator=g, device="cuda")
    gr = torch.randn(n, generator=g, device="cuda")
    m0 = torch.randn(n, generator=g, device="cuda") * 0.1
    v0 = torch.rand(n, generator=g, device="cuda") * 0.1
    lr, b1, b2, eps, wd, t = 1e-3, 0.9, 0.999, 0.01, 1e-6, 3
    step = torch.full((1,), t, dtype=torch.int32, device="cuda")

    def run(ranges):
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        stage = torch.full((rows, 40), 5.0, device="cuda", dtype=torch.bfloat16)
        stage_lo = torch.full((rows, 40), 5.0, device="cuda", dtype=torch.bfloat16)
        for lo, hi in ranges:
            segs = [(off - lo, rows, cols, stage, 40, stage_lo)] if (off < hi and lo < off + rows * cols) else []  # any overlap
            L.check(lib.spv_adam(p.data_ptr() + 4 * lo, gr.data_ptr() + 4 * lo, m.data_ptr() + 4 * lo, v.data_ptr() + 4 * lo, hi - lo,
                                 lr, b1, b2, eps, wd, 1.0, step.data_ptr(), None, len(segs), L.ll_array([s[0] for s in segs]),
                                 L.int_array([s[1] for s in segs]), L.int_array([s[2] for s in segs]),
                                 L.ptr_array([s[3] for s in segs]), L.ptr_array([s[5] for s in segs]), L.int_array([0 for _ in segs]),
                                 L.ll_array([s[4] for s in segs]), 0, _stream()), "spv_adam")
        torch.cuda.synchronize()
        return p, m, v, torch.stack([stage, stage_lo])

    pa, ma, va, sa2 = run([(0, n)])
    pb, mb, vb, sb2 = run([(0, 1000), (1000, 2048), (2048, n)])
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb) and torch.equal(sa2, sb2)
    sa, sa_lo = sa2[0], sa2[1]
    blk = pa[off:off + rows * cols].view(rows, cols)
    assert torch.equal(sa[:, :cols], blk.bfloat16())
    assert torch.equal(sa_lo[:, :cols], (blk - blk.bfloat16().float()).bfloat16())  # residual plane of the split-operand GEMM
    assert float((sa[:, cols:] - 5.0).abs().max()) == 0.0
    gd = gr.double() + wd * p0.double()
    m_ref = b1 * m0.double() + (1 - b1) * gd
    v_ref = b2 * v0.double() + (1 - b2) * gd * gd
    p_ref = p0.double() - lr / (1 - b1 ** t) * m_ref / (v_ref.sqrt() / (1 - b2 ** t) ** 0.5 + eps)
    assert float((pa.double() - p_ref).abs().max()) < 1e-6
    # ticket mode: uses *step + 1 and stores it
    step2 = torch.full((1,), t - 1, dtype=torch.int32, device="cuda")
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    p, m, v = p0.clone(), m0.clone(), v0.clone()
    L.check(lib.spv_adam(p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, b1, b2, eps, wd, 1.0, step2.data_ptr(),
                         ticket.data_ptr(), 0, None, None, None, None, None, None, None, 0, _stream()), "spv_adam")
    torch.cuda.synchronize()
    assert int(step2) == t and int(ticket) == 0 and torch.equal(p, pa)
