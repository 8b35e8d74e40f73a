"""mfa_attention_run_host (the e2e entry point bench.py times): host buffers in, host buffers out.  Checked against
the CPU oracle and against the device-pointer path, for a single problem and for batches that the library cuts into
chunks rotating over three streams (uploads, kernels and downloads of neighbouring chunks overlap)."""
import numpy as np
import pytest


def _host_run(desc, nets, types, pinned):
    import torch
    import mfa_b200 as mfa
    import oracle
    Op = mfa.AttentionOperand
    prec = desc.memoryPrecisions
    R, C, D = desc.matrixDimensions
    B = len(nets)
    host = {}
    for op, name in ((Op.Q, "Q"), (Op.K, "K"), (Op.V, "V"), (Op.dO, "dO")):
        raw = oracle.encode(np.stack([getattr(n, name) for n in nets]).astype(np.float32), int(prec[op]))
        t = torch.from_numpy(raw.view(np.int16) if raw.dtype == np.uint16 else raw)
        host[op] = t.pin_memory() if pinned else t.clone()
    shapes = {Op.O: (B, R, D), Op.L: (B, R), Op.D: (B, R), Op.dQ: (B, R, D), Op.dK: (B, C, D), Op.dV: (B, C, D)}
    for op, shape in shapes.items():
        dt = torch.float32 if prec[op] == mfa.GEMMOperandPrecision.FP32 else torch.int16
        t = torch.full(shape, float("nan") if dt == torch.float32 else -1, dtype=dt)
        host[op] = t.pin_memory() if pinned else t
    desc.runHost(types, {op: t.data_ptr() for op, t in host.items()}, device=torch.cuda.current_device())
    out = {}
    for op in shapes:
        a = host[op].numpy()
        out[op.name] = a if a.dtype == np.float32 else oracle.decode(a.view(np.uint16), int(prec[op]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("batch,R,C,D,bf16,pinned", [(1, 200, 333, 64, True, True), (5, 256, 256, 128, True, True),
                                                     (19, 130, 70, 64, False, True), (3, 64, 48, 24, None, False),
                                                     (40, 1024, 1024, 128, True, True)])
def test_run_host_matches_oracle_and_device_path(batch, R, C, D, bf16, pinned):
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention, LOG2E

    KT = mfa.AttentionKernelType
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = bf16 is not None          # None: the FP32 family
    if bf16 is not None:
        desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16 if bf16 else mfa.GEMMOperandPrecision.FP16
    desc.matrixDimensions = (R, C, D)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = batch
    prec = desc.memoryPrecisions
    nets = [oracle.Network(R, C, D, seed=100 + b, threads=8).round_inputs(int(prec[mfa.AttentionOperand.Q]),
                                                                             int(prec[mfa.AttentionOperand.dO]))
            for b in range(batch)]
    out = _host_run(desc, nets, list(KT), pinned)

    # device-pointer path on the same inputs: the chunked host path must reproduce it bit for bit (chunking only
    # changes which launch a head belongs to, never its arithmetic) -- except where split-KV engages for small grids
    inputs = {getattr(mfa.AttentionOperand, k): np.stack([getattr(n, k) for n in nets]) for k in ("Q", "K", "V", "dO")}
    dev = run_attention(desc, None, inputs=inputs, return_raw=True)
    for name in ("O", "L", "D", "dQ", "dK", "dV"):
        a, b = out[name].reshape(dev[name].shape), dev[name]
        assert np.isfinite(a).all(), name
        np.testing.assert_allclose(a, b, rtol=2e-3 if bf16 is not None else 1e-5, atol=2e-3 if bf16 is not None else 1e-5,
                                   err_msg=name)

    # and the oracle, on a few of the heads
    tol = 2e-5 if bf16 is None else 5e-2
    for b in sorted({0, batch // 2, batch - 1}):
        n = nets[b]
        O, L = n.inferenceAttention(with_L=True)
        assert np.abs(out["O"][b] - O).max() <= tol
        assert np.abs(out["L"][b] / np.float32(LOG2E) - L).max() <= (2e-5 if bf16 is None else 7e-3)
        for name, expected in (("dV", n.derivativeV()), ("dK", n.derivativeK()), ("dQ", n.derivativeQ())):
            assert np.abs(out[name][b] - expected).max() <= tol, (name, b)


@pytest.mark.gpu
def test_run_host_forward_only_leaves_other_outputs_untouched():
    import mfa_b200 as mfa
    import oracle
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    desc.matrixDimensions = (300, 300, 128)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = 12
    nets = [oracle.Network(300, 300, 128, seed=b, threads=8).round_inputs(oracle.BF16) for b in range(12)]
    out = _host_run(desc, nets, [mfa.AttentionKernelType.forward], True)
    assert np.isfinite(out["O"]).all() and np.isnan(out["dQ"]).all() and np.isnan(out["dK"]).all()
    O = nets[7].inferenceAttention()
    assert np.abs(out["O"][7] - O).max() <= 5e-3


@pytest.mark.gpu
def test_run_host_with_numa_local_buffers_and_release():
    """mfa_host_alloc / mfa_host_alloc_upload buffers (page-locked, first-touched on the GPU's NUMA node) through run_host; the caller's CPU
    affinity and current device are unchanged afterwards; mfa_release_device_resources frees the scratch and the next call
    simply allocates again."""
    import ctypes
    import os
    import torch
    import mfa_b200 as mfa
    import oracle
    Op = mfa.AttentionOperand
    B, R, C, D = 6, 256, 384, 128
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    desc.matrixDimensions = (R, C, D)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = B
    nets = [oracle.Network(R, C, D, seed=40 + b, threads=8).round_inputs(oracle.BF16) for b in range(B)]
    affinity = os.sched_getaffinity(0)
    device = torch.cuda.current_device()
    sizes = {Op.Q: B * R * D * 2, Op.K: B * C * D * 2, Op.V: B * C * D * 2, Op.O: B * R * D * 4, Op.L: B * R * 4}
    # inputs in write-combined upload buffers (mfa_host_alloc_upload), outputs in cacheable ones
    addr = {op: mfa.hostAlloc(n, device, upload=op in (Op.Q, Op.K, Op.V)) for op, n in sizes.items()}
    try:
        assert os.sched_getaffinity(0) == affinity, "mfa_host_alloc must not leave the thread re-bound"
        for op, name in ((Op.Q, "Q"), (Op.K, "K"), (Op.V, "V")):
            raw = oracle.encode(np.stack([getattr(n, name) for n in nets]).astype(np.float32), oracle.BF16)
            ctypes.memmove(addr[op], raw.ctypes.data, raw.nbytes)
        for round_ in range(2):
            ctypes.memset(addr[Op.O], 0xFF, sizes[Op.O])
            desc.runHost([mfa.AttentionKernelType.forward], addr, device=device)
            assert torch.cuda.current_device() == device
            O = np.ctypeslib.as_array((ctypes.c_float * (B * R * D)).from_address(addr[Op.O])).reshape(B, R, D)
            for b in (0, B - 1):
                assert np.abs(O[b] - nets[b].inferenceAttention()).max() <= 5e-3
            mfa.releaseDeviceResources(device)   # second round: everything is allocated afresh
    finally:
        for a in addr.values():
            mfa.hostFree(a)
    node = mfa.bindThreadToDevice(device)
    try:
        assert node >= -1 and len(os.sched_getaffinity(0)) >= 1
    finally:
        os.sched_setaffinity(0, affinity)


@pytest.mark.gpu
def test_one_process_drives_two_gpus():
    """The API lets one process use several devices (run_host takes the device; encode runs on the current one): kernel
    attributes, SM counts, scratch and workspaces are all per device.  Skipped on a single-GPU box."""
    import torch
    import mfa_b200 as mfa
    import oracle
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs in one process")
    KT = mfa.AttentionKernelType
    for R, C, D, batch in ((256, 256, 128, 3), (4096, 4096, 128, 1)):   # plain and split-KV grids
        desc = mfa.AttentionDescriptor()
        desc.lowPrecisionInputs = True
        desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
        desc.matrixDimensions = (R, C, D)
        desc.transposeState = (False, False, False, False)
        desc.batchCount = batch
        nets = [oracle.Network(R, C, D, seed=70 + b, threads=16).round_inputs(oracle.BF16) for b in range(batch)]
        types = list(KT) if R <= 256 else [KT.forward]
        for device in (0, 1, 0):
            torch.cuda.set_device(0)
            prev = torch.cuda.current_device()
            Op = mfa.AttentionOperand
            prec = desc.memoryPrecisions
            host = {}
            for op, name in ((Op.Q, "Q"), (Op.K, "K"), (Op.V, "V"), (Op.dO, "dO")):
                raw = oracle.encode(np.stack([getattr(n, name) for n in nets]).astype(np.float32), int(prec[op]))
                host[op] = torch.from_numpy(raw.view(np.int16)).pin_memory()
            for op, shape in {Op.O: (batch, R, D), Op.L: (batch, R), Op.D: (batch, R), Op.dQ: (batch, R, D),
                              Op.dK: (batch, C, D), Op.dV: (batch, C, D)}.items():
                host[op] = torch.full(shape, float("nan"), dtype=torch.float32).pin_memory()
            desc.runHost(types, {op: t.data_ptr() for op, t in host.items()}, device=device)
            assert torch.cuda.current_device() == prev, "run_host must restore the caller's device"
            O = nets[batch - 1].inferenceAttention()
            assert np.abs(host[Op.O][batch - 1].numpy() - O).max() <= 5e-3, (device, R)
            if len(types) == 3:
                dQ = nets[0].derivativeQ()
                assert np.abs(host[Op.dQ][0].numpy() - dQ).max() <= 5e-2, device


@pytest.mark.gpu
def test_batches_beyond_the_grid_limit_are_sliced():
    """batch_count > 16384 problems per encode(): kernels that carry the batch in gridDim.y (limit 65535) are launched
    over slices of the batch; every slice must land at the right offset."""
    import torch
    import mfa_b200 as mfa
    import oracle
    from tests.attention_harness import run_attention
    batch, R, C, D = 16384 + 37, 16, 24, 16
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.FP16
    desc.matrixDimensions = (R, C, D)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = batch
    base = oracle.Network(R, C, D, seed=5).round_inputs(oracle.FP16)
    rng = np.random.default_rng(0)
    scale = (1.0 + 0.25 * rng.standard_normal(batch)).astype(np.float16).astype(np.float32)[:, None, None]
    Op = mfa.AttentionOperand
    inputs = {Op.Q: np.broadcast_to(base.Q, (batch, R, D)).copy(), Op.K: np.broadcast_to(base.K, (batch, C, D)).copy(),
              Op.V: oracle.roundtrip(base.V[None] * scale, oracle.FP16), Op.dO: np.broadcast_to(base.dO, (batch, R, D)).copy()}
    out = run_attention(desc, None, inputs=inputs)
    O = base.inferenceAttention()
    # same Q and K everywhere, V scaled per problem: O[b] = scale'[b] * O (V was re-rounded, so compare against the
    # rounded per-problem V through linearity in V for a few problems on both sides of the slice boundary)
    for b in (0, 1, 16383, 16384, 16385, batch - 1):
        net = oracle.Network(R, C, D, seed=5).round_inputs(oracle.FP16)
        net.V = inputs[Op.V][b]
        assert np.abs(out["O"][b] - net.inferenceAttention()).max() <= 5e-3, b
        assert np.abs(out["dQ"][b] - net.derivativeQ()).max() <= 5e-2, b
    assert np.isfinite(out["dV"]).all() and np.isfinite(out["dK"]).all()
