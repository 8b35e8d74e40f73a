"""Single-head latency of the three kernels, device-timed two ways: an eager launch loop (includes whatever the host
cannot hide) and a CUDA graph of the same launches (the launch-bound inner loop captured, as a serving stack would run
it).  Where split-KV engages, the forward is two launches (attention + combine kernel).
Usage (GPU box):  python scripts/bench_single.py"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mfa_b200 as mfa  # noqa: E402

KT, Op, P = mfa.AttentionKernelType, mfa.AttentionOperand, mfa.GEMMOperandPrecision
WORK = {KT.forward: (2, 4), KT.backwardQuery: (3, 6), KT.backwardKeyValue: (4, 8)}


def time_kernel(kernel, constants, ptrs, launches=20, replays=10):
    stream = torch.cuda.Stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        for _ in range(5):
            kernel.encode(constants, ptrs, stream.cuda_stream)
        stream.synchronize()
        a.record(stream)
        for _ in range(launches * replays):
            kernel.encode(constants, ptrs, stream.cuda_stream)
        b.record(stream)
        stream.synchronize()
        eager_us = a.elapsed_time(b) * 1e3 / (launches * replays)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for _ in range(launches):
                kernel.encode(constants, ptrs, stream.cuda_stream)
        for _ in range(3):
            graph.replay()
        stream.synchronize()
        a.record(stream)
        for _ in range(replays):
            graph.replay()
        b.record(stream)
        stream.synchronize()
        graph_us = a.elapsed_time(b) * 1e3 / (launches * replays)
    return eager_us, graph_us


def run(N, D, precision, H=1):
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.inputPrecisionOverride = precision
    desc.matrixDimensions = (N, N, D)
    desc.transposeState = (False,) * 4
    desc.batchCount = H
    dt = torch.bfloat16 if precision == P.BF16 else torch.float16
    bufs = {op: torch.randn(H, N, D, device="cuda").to(dt) for op in (Op.Q, Op.K, Op.V, Op.dO)}
    for op in (Op.O, Op.dQ, Op.dK, Op.dV):
        bufs[op] = torch.empty(H, N, D, device="cuda")
    for op in (Op.L, Op.D):
        bufs[op] = torch.empty(H, N, device="cuda")
    ptrs = {op: t.data_ptr() for op, t in bufs.items()}
    c = mfa.FunctionConstantValues()
    desc.setFunctionConstants(c)
    out = {"N": N, "D": D, "dtype": precision.name, "heads": H}
    for t in KT:
        if D > 128 and t != KT.forward:
            continue
        k = mfa.AttentionKernel(desc.kernelDescriptor(t))
        launches = k.launchCount(c)
        eager_us, graph_us = time_kernel(k, c, ptrs)
        fma, gemm = WORK[t]
        out[t.name] = {"launches": launches, "eager_us": round(eager_us, 2), "graph_us": round(graph_us, 2),
                       "tflops_graph": round(gemm * N * N * D * H / graph_us / 1e6, 1),
                       "ginstrs_graph": round((fma * D + 5) * N * N * H / graph_us / 1e3, 1)}
    return out


if __name__ == "__main__":
    for N, D, prec in ((4096, 128, P.BF16), (2048, 64, P.FP16), (8192, 256, P.BF16), (8192, 128, P.BF16),
                       (2048, 128, P.BF16), (1024, 128, P.BF16)):
        print(json.dumps(run(N, D, prec)), flush=True)
