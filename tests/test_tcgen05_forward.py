"""Parity of the tensor-core forward (TMA + tcgen05 + TMEM) with the CPU oracle.

The oracle runs on the inputs AFTER rounding to the kernel's 16-bit memory format, so the comparison
isolates the kernel's own arithmetic.  Stated tolerances (north_star: "within 1e-3 relative"):
  O : relative RMS error  rms(O - O_ref) / rms(O_ref) <= 3e-4 for FP16 and <= 2e-3 for BF16.  These are the
      quantisation floors of P, the A operand of O += P V, which is rounded to the MMA input type: round-to-nearest with
      s significant bits has a relative error uniform in +-2^-s / (1 + f), rms 2^-s / sqrt(6) -- 1.99e-4 for FP16
      (s = 11), 1.59e-3 for BF16 (s = 8) -- and the row sum does not average it away relative to O.  Measured
      (profiles/r2_parity.jsonl): 1.98e-4 and 1.59e-3 at N = 4096, D = 128.  And element-wise
      |err| <= eps_P * max|V| + 1e-5 with eps_P = 2^-8 (bf16) or 2^-10 (fp16): P is rounded to the 16-bit MMA
      input type before O += P V, so each element carries at most half an ulp of P times the V it multiplies
      (the bound is reached when C is tiny and nothing averages out);
  L : |err| <= 1e-3 absolute in natural-log units (FP32 L); 7e-3 when L is stored as FP16 (reference's bar)
and always within the reference's own mixed-precision bars O 5e-2 / L 7e-3 (SquareAttentionTest.swift:539-546)."""
import numpy as np
import pytest


def _descriptor(R, C, D, bf16, lowMid=False, batch=1):
    import mfa_b200 as mfa
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.lowPrecisionIntermediates = lowMid
    desc.matrixDimensions = (R, C, D)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = batch
    if bf16:
        desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    return desc


def _run_and_check(R, C, D, bf16, seed, lowMid=False, threads=8):
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check

    desc = _descriptor(R, C, D, bf16, lowMid)
    kd = desc.kernelDescriptor(mfa.AttentionKernelType.forward)
    assert kd.backend == mfa.Backend.tcgen05, "heuristic should pick the tensor-core family here"
    net = oracle.Network(R, C, D, seed=seed, threads=threads).round_inputs(oracle.BF16 if bf16 else oracle.FP16)
    out = run_attention(desc, net, types=[mfa.AttentionKernelType.forward])
    O, L = net.inferenceAttention(with_L=True)
    errO = check_O(O, out["O"], net.V, bf16)
    errL = check(L, out["L"], 7e-3 if lowMid else 1e-3, "L")
    return errO, errL


def check_O(O, actual, V, bf16, name="O"):
    from tests.attention_harness import check
    tolO = (2.0 ** -8 if bf16 else 2.0 ** -10) * float(np.abs(V).max()) + 1e-5
    errO = check(O, actual, min(tolO, 5e-2), name)
    rel_rms = float(np.sqrt(np.mean((actual - O) ** 2)) / max(np.sqrt(np.mean(O ** 2)), 1e-30))
    bound = 2e-3 if bf16 else 3e-4
    assert rel_rms <= bound, f"{name}: relative RMS error {rel_rms:.3e} > {bound}"
    return errO


@pytest.mark.gpu
@pytest.mark.parametrize("bf16", [True, False], ids=["bf16", "fp16"])
@pytest.mark.parametrize("R,C,D", [
    (256, 256, 128), (128, 128, 64), (512, 384, 128), (256, 640, 64),   # aligned
    (200, 333, 128), (77, 129, 64), (1, 1, 8), (300, 17, 80), (129, 257, 72), (40, 500, 16),  # ragged edges
    (1024, 1024, 128), (640, 1280, 96),
    (256, 256, 256), (200, 333, 192), (384, 512, 136), (130, 70, 256), (1024, 1024, 256),   # 128 < D <= 256 kernel
])
def test_forward_matches_oracle(R, C, D, bf16):
    _run_and_check(R, C, D, bf16, seed=R * 7 + C * 3 + D)


SPLIT_KV_CASES = [(4096, 4096, 128, True),   # 16 items x 8 splits: the headline single head
                  (256, 2048, 64, False),    # 1 item x 4 splits
                  (300, 2000, 128, True),    # ragged rows and a ragged last key block
                  (512, 1536, 96, True),     # 12 key blocks -> 3 splits
                  (1, 4096, 128, False),     # a single query row
                  (2048, 2048, 64, True)]    # BASELINE configs[2] shape


@pytest.mark.gpu
@pytest.mark.parametrize("R,C,D,bf16", SPLIT_KV_CASES)
def test_split_kv_small_grids(R, C, D, bf16):
    """Few (head, tile pair) items: the key axis is split across SMs.  Normalised partials go to the library's workspace
    and the combine kernel merges them (2 launches).  Must match the oracle, also when run back to back."""
    import mfa_b200 as mfa
    desc = _descriptor(R, C, D, bf16)
    kernel = mfa.AttentionKernel(desc.kernelDescriptor(mfa.AttentionKernelType.forward))
    constants = mfa.FunctionConstantValues()
    desc.setFunctionConstants(constants)
    assert kernel.launchCount(constants) == 2, "split-KV should engage for this grid"
    _run_and_check(R, C, D, bf16, seed=R + C + D)
    _run_and_check(R, C, D, bf16, seed=R + C + D + 1)


@pytest.mark.gpu
def test_split_kv_batched_heads_and_fp16_L():
    """Split-KV with several heads in one launch (item -> (head, tile, split)) and FP16 L storage."""
    import mfa_b200 as mfa
    H, N, D = 3, 1024, 128
    desc = _descriptor(N, N, D, True, lowMid=True, batch=H)
    kernel = mfa.AttentionKernel(desc.kernelDescriptor(mfa.AttentionKernelType.forward))
    constants = mfa.FunctionConstantValues()
    desc.setFunctionConstants(constants)
    assert kernel.launchCount(constants) == 2
    _check_batched_cluster(desc, H, N, D)


def _check_batched_cluster(desc, H, N, D):
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check
    nets = [oracle.Network(N, N, D, seed=100 + h, threads=8).round_inputs(oracle.BF16) for h in range(H)]
    Op = mfa.AttentionOperand
    inputs = {Op.Q: np.stack([n.Q for n in nets]), Op.K: np.stack([n.K for n in nets]),
              Op.V: np.stack([n.V for n in nets])}
    out = run_attention(desc, None, types=[mfa.AttentionKernelType.forward], inputs=inputs)
    for h, net in enumerate(nets):
        O, L = net.inferenceAttention(with_L=True)
        check_O(O, out["O"][h], net.V, True, name=f"O[head {h}]")
        check(L, out["L"][h], 7e-3, f"L[head {h}]")


@pytest.mark.gpu
def test_forward_fp16_L_storage():
    """lowPrecisionIntermediates: L is stored as FP16 (AttentionDescriptor+Precisions.swift:81-87)."""
    _run_and_check(256, 256, 128, True, seed=5, lowMid=True)
    _run_and_check(192, 200, 64, False, seed=6, lowMid=True)


@pytest.mark.gpu
def test_config2_full_size_bf16_n4096_d128():
    """BASELINE.json configs[1]: single-head forward bf16 N=4096 D=128, against the (row-parallel) oracle."""
    errO, errL = _run_and_check(4096, 4096, 128, True, seed=0)
    print(f"config2 max|dO|={errO:.3e} max|dL|={errL:.3e}")


@pytest.mark.gpu
def test_config4_large_head_bf16_n8192_d256():
    """BASELINE.json configs[3]: the large-D path, forward bf16 N=8192 D=256 (one tile per CTA, O in 256 TMEM columns)."""
    errO, errL = _run_and_check(8192, 8192, 256, True, seed=4, threads=64)
    print(f"config4 max|dO|={errO:.3e} max|dL|={errL:.3e}")


@pytest.mark.gpu
def test_adversarial_growing_max_forces_rescale():
    """Scores that keep growing along the key axis force the (normally rare) O-rescale path every block."""
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check

    R, C, D = 256, 1024, 64
    net = oracle.Network(R, C, D, seed=11, threads=8)
    ramp = np.linspace(0.0, 6.0, C, dtype=np.float32)[:, None]
    net.K = net.K + ramp * np.sign(net.Q.mean(axis=0, keepdims=True) + 1e-3)
    net.Q = np.abs(net.Q) * np.sign(net.Q.mean(axis=0, keepdims=True) + 1e-3)
    net.round_inputs(oracle.BF16)
    desc = _descriptor(R, C, D, True)
    out = run_attention(desc, net, types=[mfa.AttentionKernelType.forward])
    O, L = net.inferenceAttention(with_L=True)
    check_O(O, out["O"], net.V, True)
    check(L, out["L"], 2e-3, "L")


@pytest.mark.gpu
@pytest.mark.parametrize("C", [512, 417, 33])
def test_adversarial_growing_max_large_head(C):
    """Same adversarial construction on the 128 < D <= 256 kernel, whose rows are split over two warps that take the
    rescale decision jointly (named barrier with OR reduction) and rescale half of the O columns each; the ragged
    column counts put the masked tail into one warp's half only."""
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check

    R, D = 200, 256
    net = oracle.Network(R, C, D, seed=13, threads=8)
    ramp = np.linspace(0.0, 4.0, C, dtype=np.float32)[:, None]
    net.K = net.K + ramp * np.sign(net.Q.mean(axis=0, keepdims=True) + 1e-3)
    net.Q = np.abs(net.Q) * np.sign(net.Q.mean(axis=0, keepdims=True) + 1e-3)
    net.K[C // 2 + 5] = net.Q[7] * 1.5     # a late jump for row 7
    net.round_inputs(oracle.BF16)
    desc = _descriptor(R, C, D, True)
    out = run_attention(desc, net, types=[mfa.AttentionKernelType.forward])
    O, L = net.inferenceAttention(with_L=True)
    check_O(O, out["O"], net.V, True)
    check(L, out["L"], 2e-3, "L")


@pytest.mark.gpu
@pytest.mark.parametrize("R,C,D", [(256, 384, 128), (200, 136, 64), (264, 520, 256), (8, 8, 8), (136, 1000, 192),
                                   (1024, 1024, 128)])
@pytest.mark.parametrize("mask", range(1, 16))
def test_forward_transposed_operands(R, C, D, mask):
    """Every combination of transposed Q, K, V, O (stored [D][seq], AttentionKernel.swift:189-195;
    RectangularAttentionTest.swift:88-138) on the layout-generic tensor-core kernel: transposed Q / K tiles are MN-major
    MMA operands, a transposed V is K-major, a transposed O is stored straight from registers."""
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check

    if (R, C, D) == (1024, 1024, 128) and mask not in (5, 10, 15):
        pytest.skip("large shape: three masks only")
    bf16 = mask % 2 == 1
    desc = _descriptor(R, C, D, bf16)
    desc.transposeState = tuple(bool(mask & (1 << i)) for i in range(4))
    kd = desc.kernelDescriptor(mfa.AttentionKernelType.forward)
    assert kd.backend == mfa.Backend.tcgen05 and kd.blockDimensions[:2] == (128, 128)
    net = oracle.Network(R, C, D, seed=mask + R, threads=8)
    net.round_inputs(oracle.BF16 if bf16 else oracle.FP16)
    out = run_attention(desc, net, types=[mfa.AttentionKernelType.forward])
    O, L = net.inferenceAttention(with_L=True)
    check_O(O, out["O"], net.V, bf16)
    check(L, out["L"], 1e-3, "L")


@pytest.mark.gpu
def test_batched_heads_are_independent_problems():
    """batch extension: problem b of the batch equals the single-head run on the same tensors; and the
    softmax identity O == 1 when V == 1 holds at the full N=4096 (size-independent property)."""
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, check

    R = C = 512
    D = 128
    nets = [oracle.Network(R, C, D, seed=s, threads=8).round_inputs(oracle.BF16) for s in (21, 22, 23)]
    desc = _descriptor(R, C, D, True, batch=3)
    Op = mfa.AttentionOperand
    inputs = {Op.Q: np.stack([n.Q for n in nets]), Op.K: np.stack([n.K for n in nets]),
              Op.V: np.stack([n.V for n in nets])}
    out = run_attention(desc, None, types=[mfa.AttentionKernelType.forward], inputs=inputs)
    for b, n in enumerate(nets):
        O, L = n.inferenceAttention(with_L=True)
        check_O(O, out["O"][b], n.V, True, f"O[{b}]")
        check(L, out["L"][b], 1e-3, f"L[{b}]")

    N = 4096
    big = oracle.Network(N, N, D, seed=3).round_inputs(oracle.BF16)
    big.V = np.ones_like(big.V)
    out = run_attention(_descriptor(N, N, D, True), big, types=[mfa.AttentionKernelType.forward])
    # rows of P sum to 1 -> O == 1 up to the 16-bit rounding of P (relative 2^-9, averaged over the row)
    assert np.abs(out["O"] - 1.0).max() < 2e-3
