"""Runs a GEMMDescriptor through the library on the current GPU the way the reference's GEMM tests do
(Tests/FlashAttentionTests/GEMM/AdversarialShapeTest.swift:94-239): operands are FP32 arrays laid out with the
descriptor's leading dimensions, rounded to their memory precision on upload, and the product is checked against a
float64 product of the same FP32 arrays -- the unrounded values, as the reference's CPU loop uses them -- under the
reference's createTolerance (:288-336)."""
import numpy as np

import mfa_b200 as mfa

P = mfa.GEMMOperandPrecision


def torch_dtype(precision):
    import torch
    return {P.FP32: torch.float32, P.FP16: torch.float16, P.BF16: torch.bfloat16}[P(precision)]


def stored_shapes(M, N, K, transpose):
    """(rows, columns) of A, B and C as stored (chooseTrailingBlockDimension / the leading dimension's minimum)."""
    tA, tB = transpose
    return ((K, M) if tA else (M, K)), ((N, K) if tB else (K, N)), (M, N)


def leading_dimensions(desc):
    c = mfa.GEMMFunctionConstantValues()
    desc.setFunctionConstants(c)
    return c.leadingDimensions


def device_buffer(array, precision, byte_offset=0):
    """A flat device copy of `array` (FP32) in `precision`, starting `byte_offset` bytes into its allocation.
    Returns (keep-alive tensor, pointer, view of the data)."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(array, dtype=np.float32).reshape(-1))
    dtype = torch_dtype(precision)
    element = torch.empty((), dtype=dtype).element_size()
    assert byte_offset % element == 0
    pad = byte_offset // element
    storage = torch.zeros(flat.numel() + pad + 8, dtype=dtype, device="cuda")
    view = storage[pad:pad + flat.numel()]
    view.copy_(flat.to(dtype))
    return storage, view.data_ptr(), view


def reference_product(A, B, prevC, desc):
    """float64 C (+ prevC) over the [batch, rows, leading] arrays, addressed as AdversarialShapeTest.swift:211-236."""
    M, N, K = desc.matrixDimensions
    tA, tB = desc.transposeState
    out = []
    for b in range(A.shape[0]):
        a = A[b, :K, :M].T if tA else A[b, :M, :K]
        bb = B[b, :N, :K].T if tB else B[b, :K, :N]
        c = a.astype(np.float64) @ bb.astype(np.float64)
        if desc.loadPreviousC:
            c = c + prevC[b, :M, :N].astype(np.float64)
        out.append(c)
    return np.stack(out)


def create_tolerance(precisions, K):
    """createTolerance, AdversarialShapeTest.swift:288-336."""
    A, B, C = (P(p) for p in precisions)
    noise = float(np.sqrt(K))
    tol = 3e-7
    if A == P.FP16 or B == P.FP16:
        tol = max(tol, 1e-5)
        tol = max(tol, 1e-3 / noise)
    if C == P.FP16:
        tol = max(tol, 3e-4)
    if A == B == C == P.FP16:
        tol = max(tol, 3e-3)
        tol = max(tol, 1e-5 * K)
    if P.BF16 in (A, B, C):
        tol = max(tol, 2e-2 if K < 1000 else 5e-3)
    tol += 2.0 ** -8 if C == P.BF16 else (2.0 ** -10 if C == P.FP16 else 2.0 ** -22)
    return tol


def run_gemm(desc, A, B, prevC, offsets=(0, 0, 0), stream=None, kernel=None):
    """Encode `desc` on A, B, C = prevC ([batch, rows, leading] FP32 arrays); returns C as FP32 [batch, M, ldc] and the
    kernel object used.  `offsets`: byte offsets of the three base pointers."""
    import torch
    precisions = desc.memoryPrecisions
    keep = []
    pointers = []
    views = []
    for array, precision, offset in zip((A, B, prevC), precisions, offsets):
        storage, ptr, view = device_buffer(array, precision, offset)
        keep.append(storage)
        pointers.append(ptr)
        views.append(view)
    if kernel is None:
        mfa.GEMMKernel.register(desc)
        kernel = mfa.GEMMKernel.cached(desc)
    constants = mfa.GEMMFunctionConstantValues()
    desc.setFunctionConstants(constants)
    s = stream if stream is not None else torch.cuda.current_stream()
    kernel.encode(constants, pointers, stream=s.cuda_stream)
    s.synchronize()
    C = views[2].float().cpu().numpy().reshape(prevC.shape)
    return C, kernel


def random_problem(desc, rng):
    """FP32 A, B, previous C filled the reference's way: uniform [0, 1) / sqrt(K) (AdversarialShapeTest.swift:108-124),
    including the padding columns between the width and the leading dimension."""
    M, N, K = desc.matrixDimensions
    batch = max(1, desc.batchDimension)
    lda, ldb, ldc = leading_dimensions(desc)
    (ra, _), (rb, _), (rc, _) = stored_shapes(M, N, K, desc.transposeState)
    f = 1.0 / np.sqrt(K)
    A = (rng.random((batch, ra, lda), dtype=np.float32) * f).astype(np.float32)
    B = (rng.random((batch, rb, ldb), dtype=np.float32) * f).astype(np.float32)
    C = (rng.random((batch, rc, ldc), dtype=np.float32) * f).astype(np.float32)
    return A, B, C


def max_distance(C, expected, desc):
    M, N, _ = desc.matrixDimensions
    return float(np.abs(C[:, :M, :N].astype(np.float64) - expected).max())
