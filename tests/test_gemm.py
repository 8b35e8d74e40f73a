"""GEMM on the B200: the reference's two GEMM test suites (LaplacianTest.swift, AdversarialShapeTest.swift) plus the
cases specific to the tcgen05 kernel -- large products against torch, ragged edges, batches, the staging path for
unaligned operands, loadPreviousC in place, streams and CUDA-graph capture."""
import numpy as np
import pytest

from tests import gemm_harness as H

# LaplacianTest.swift:6-25
LAPLACIAN_SIZES = [7, 8, 9, 10, 15, 16, 17, 18, 23, 24, 25, 31, 32, 33, 47, 48, 49, 63, 64, 65, 103, 104, 112,
                   126, 127, 128, 129, 130, 131, 135, 136, 137, 143, 144, 145, 151, 152, 153]
LAPLACIAN_TRANSPOSES = [(False, False), (False, True), (True, False)]


def _gemm(M, N, K, precisions, transpose=(False, False), load_previous=False, leading=None, batch=1):
    import mfa_b200 as mfa
    d = mfa.GEMMDescriptor()
    d.matrixDimensions = (M, N, K)
    d.memoryPrecisions = tuple(precisions)
    d.transposeState = tuple(transpose)
    d.loadPreviousC = load_previous
    d.leadingDimensions = leading
    d.batchDimension = batch
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["FP32", "FP16", "BF16"])
@pytest.mark.parametrize("transpose", LAPLACIAN_TRANSPOSES)
def test_laplacian(precision, transpose):
    """LaplacianTest.swift:57-290: a periodic 1-D Laplacian times a random matrix (the operands swap when A is
    transposed), every entry within the reference's per-precision threshold."""
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    p = P[precision]
    threshold = {P.FP32: 1e-5, P.FP16: 5e-3, P.BF16: 5e-2}[p]
    rng = np.random.default_rng(17)
    for n in LAPLACIAN_SIZES:
        L = np.zeros((n, n), np.float32)
        for i in range(n):
            L[i, i] = -2
            L[i, (i + n - 1) % n] = 1
            L[i, (i + 1) % n] = 1
        R = rng.random((n, n), dtype=np.float32)
        A, B = (R, L) if transpose[0] else (L, R)
        d = _gemm(n, n, n, (p, p, p), transpose)
        expected = H.reference_product(A[None], B[None], None, d)
        C, kernel = H.run_gemm(d, A[None], B[None], np.zeros((1, n, n), np.float32))
        assert ("tcgen05" in kernel.sourceName()) == (p != P.FP32)
        err = H.max_distance(C, expected, d)
        assert err < threshold, (n, err)


def _adversarial_cases(count, seed):
    """AdversarialShapeTest.swift:7-65: cubed-uniform shapes x 1000, random precisions per operand, loadPreviousC,
    transposes, and (half of the time) leading dimensions padded by 0..63."""
    rng = np.random.default_rng(seed)
    cases = []
    for _ in range(count):
        dims = (rng.random(3) ** 3 * 1000).astype(np.int64)
        dims[dims == 0] = 1
        M, N, K = (int(x) for x in dims)
        precisions = tuple(int(x) for x in rng.integers(0, 3, 3))
        load_previous = bool(rng.integers(0, 2))
        transpose = (bool(rng.integers(0, 2)), bool(rng.integers(0, 2)))
        leading = (M if transpose[0] else K, K if transpose[1] else N, N)
        if rng.integers(0, 2):
            leading = tuple(int(x + rng.integers(0, 64)) for x in leading)
        cases.append((M, N, K, precisions, load_previous, transpose, leading))
    return cases


ADVERSARIAL = _adversarial_cases(120, seed=20261017)


@pytest.mark.gpu
def test_adversarial_shapes():
    """120 seeded trials; each meets createTolerance against float64, and C's padding columns stay untouched."""
    import mfa_b200 as mfa
    rng = np.random.default_rng(5)
    tensor_core = 0
    failures = []
    for i, (M, N, K, precisions, load_previous, transpose, leading) in enumerate(ADVERSARIAL):
        d = _gemm(M, N, K, precisions, transpose, load_previous, leading)
        A, B, prev = H.random_problem(d, rng)
        C, kernel = H.run_gemm(d, A, B, prev)
        expected = H.reference_product(A, B, prev, d)
        err, tol = H.max_distance(C, expected, d), H.create_tolerance(precisions, K)
        tc = mfa.GEMMKernelDescriptor(d).backend == mfa.Backend.tcgen05
        tensor_core += tc
        assert ("tcgen05" in kernel.sourceName()) == tc
        ldc = leading[2]
        if ldc > N:
            import torch
            rounded = torch.from_numpy(prev[:, :M, N:].copy()).to(H.torch_dtype(precisions[2])).float().numpy()
            assert np.array_equal(C[:, :M, N:], rounded), ("padding of C was written", i)
        if not err < tol:
            failures.append((i, M, N, K, precisions, load_previous, transpose, leading, err, tol))
    assert not failures, failures
    assert tensor_core >= 10   # the 16-bit draws, unaligned leading dimensions included, reach the tensor cores


@pytest.mark.gpu
@pytest.mark.parametrize("transpose", [(False, False), (False, True), (True, False), (True, True)])
def test_tcgen05_4096_against_torch(transpose):
    import torch
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    M = N = K = 4096
    torch.manual_seed(3)
    a = torch.randn(K, M, device="cuda").to(torch.bfloat16) if transpose[0] else \
        torch.randn(M, K, device="cuda").to(torch.bfloat16)
    b = torch.randn(N, K, device="cuda").to(torch.bfloat16) if transpose[1] else \
        torch.randn(K, N, device="cuda").to(torch.bfloat16)
    c = torch.empty(M, N, device="cuda", dtype=torch.float32)
    d = _gemm(M, N, K, (P.BF16, P.BF16, P.FP32), transpose)
    k = mfa.GEMMKernel.cached(d)
    assert k.sourceName().startswith("gemm_tcgen05")
    consts = mfa.GEMMFunctionConstantValues()
    d.setFunctionConstants(consts)
    k.encode(consts, [a.data_ptr(), b.data_ptr(), c.data_ptr()], stream=torch.cuda.current_stream().cuda_stream)
    la = a.float().T if transpose[0] else a.float()
    lb = b.float().T if transpose[1] else b.float()
    ref = torch.matmul(la, lb)   # FP32 (TF32 is off by default for torch.matmul)
    torch.cuda.synchronize()
    rel = float((c - ref).abs().max() / ref.abs().max())
    assert rel < 1e-4, rel


def _check_tc(d, rng, offsets=(0, 0, 0)):
    import mfa_b200 as mfa
    A, B, prev = H.random_problem(d, rng)
    C, kernel = H.run_gemm(d, A, B, prev, offsets=offsets)
    assert kernel.sourceName().startswith("gemm_tcgen05")
    assert mfa.GEMMKernelDescriptor(d).backend == mfa.Backend.tcgen05
    # against the product of the rounded inputs: what the tensor cores see
    import torch
    r = [torch.from_numpy(x).to(H.torch_dtype(p)).float().numpy() for x, p in zip((A, B, prev), d.memoryPrecisions)]
    expected = H.reference_product(r[0], r[1], r[2], d)
    err = H.max_distance(C, expected, d)
    tol = {0: 2e-5, 1: 2e-3, 2: 1.6e-2}[int(d.memoryPrecisions[2])] * max(1.0, float(np.abs(expected).max()))
    assert err < tol, (d.matrixDimensions, d.transposeState, err, tol)


EDGE_SHAPES = [(1, 1, 1), (127, 255, 63), (129, 257, 65), (200, 300, 17), (64, 96, 8), (300, 520, 200), (1000, 33, 130)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", EDGE_SHAPES)
@pytest.mark.parametrize("transpose", [(False, False), (False, True), (True, False), (True, True)])
def test_tcgen05_ragged_edges(shape, transpose):
    """M, N, K off the 128 / 256 / 64 tile grid and K < 64; leading dimensions stay multiples of 8 where the shape
    allows, so most of these go through TMA without staging."""
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    M, N, K = shape
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    leading = tuple((x + 7) // 8 * 8 for x in (M if transpose[0] else K, K if transpose[1] else N, N))
    for precisions in ((P.BF16, P.BF16, P.FP32), (P.FP16, P.FP16, P.FP16)):
        _check_tc(_gemm(M, N, K, precisions, transpose, leading=leading), rng)


@pytest.mark.gpu
def test_tcgen05_batch():
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    rng = np.random.default_rng(11)
    for transpose in ((False, False), (True, True)):
        d = _gemm(192, 320, 136, (P.BF16, P.BF16, P.BF16), transpose, batch=5)
        k = mfa.GEMMKernel.cached(d)
        c = mfa.GEMMFunctionConstantValues()
        d.setFunctionConstants(c)
        assert c.batchCount == 5 and k.gridSize(c) == 2 * 2 * 5
        _check_tc(d, rng)
    # unaligned leading dimensions with a batch: the staged copy keeps the problems back to back
    d = _gemm(100, 130, 70, (P.FP16, P.FP16, P.FP32), (False, True), leading=(75, 77, 131), batch=3)
    _check_tc(d, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("transpose", [(False, False), (False, True), (True, False), (True, True)])
def test_tcgen05_staging(transpose):
    """lda / ldb not multiples of 8, and base pointers 2 bytes off 16-byte alignment: the operands are staged."""
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    rng = np.random.default_rng(23)
    M, N, K = 257, 190, 333
    base = (M if transpose[0] else K, K if transpose[1] else N, N)
    unaligned = tuple(x + 1 if (x + 1) % 8 else x + 2 for x in base)   # leading dimensions that are not multiples of 8
    d = _gemm(M, N, K, (P.BF16, P.BF16, P.FP32), transpose, leading=unaligned)
    c = mfa.GEMMFunctionConstantValues()
    d.setFunctionConstants(c)
    assert mfa.GEMMKernel.cached(d).launchCount(c) == 3
    _check_tc(d, rng)
    aligned = _gemm(M, N, K, (P.BF16, P.BF16, P.FP32), transpose,
                    leading=tuple((x + 7) // 8 * 8 for x in base))
    _check_tc(aligned, rng, offsets=(2, 2, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("precision_C", ["FP32", "FP16", "BF16"])
def test_tcgen05_load_previous_C_in_place(precision_C):
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    rng = np.random.default_rng(31)
    for leading in (None, (136, 264, 263)):
        d = _gemm(300, 260, 130, (P.FP16, P.FP16, P[precision_C]), load_previous=True, leading=leading)
        _check_tc(d, rng)


@pytest.mark.gpu
def test_source_name_follows_backend():
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    for a in P:
        for b in P:
            for c in P:
                for t in ((False, False), (False, True), (True, False), (True, True)):
                    d = _gemm(64, 64, 64, (a, b, c), t)
                    tc = mfa.GEMMKernelDescriptor(d).backend == mfa.Backend.tcgen05
                    assert mfa.GEMMKernel.cached(d).sourceName().startswith("gemm_tcgen05" if tc else "gemm_simt_fp32")


@pytest.mark.gpu
def test_tcgen05_non_default_stream_and_graph_capture():
    import torch
    import mfa_b200 as mfa
    P = mfa.GEMMOperandPrecision
    M, N, K = 512, 768, 320
    torch.manual_seed(0)
    a = torch.randn(M, K, device="cuda").half()
    b = torch.randn(K, N, device="cuda").half()
    c = torch.zeros(M, N, device="cuda")
    d = _gemm(M, N, K, (P.FP16, P.FP16, P.FP32), leading=(K + 1, N, N))   # unaligned lda: staging workspace too
    k = mfa.GEMMKernel.cached(d)
    a_padded = torch.zeros(M, K + 1, device="cuda").half()
    a_padded[:, :K] = a
    consts = mfa.GEMMFunctionConstantValues()
    d.setFunctionConstants(consts)
    ref = (a.double() @ b.double())
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        k.encode(consts, [a_padded.data_ptr(), b.data_ptr(), c.data_ptr()], stream=stream.cuda_stream)
    stream.synchronize()
    assert float((c.double() - ref).abs().max()) < 1e-3
    # capture on the stream of the warm-up encode above (the staging workspace belongs to a (device, stream) pair)
    c.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        k.encode(consts, [a_padded.data_ptr(), b.data_ptr(), c.data_ptr()], stream=stream.cuda_stream)
    c.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert float((c.double() - ref).abs().max()) < 1e-3
