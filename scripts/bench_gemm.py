"""Times the tcgen05 GEMM against torch.matmul on one GPU and appends one JSON line per configuration.

Configurations: bf16 and fp16 inputs, M = N = K = 4096 and 8192, the four transpose states, FP32 and 16-bit C.
For each, both libraries run on the same tensors in the same process, alternating, with CUDA events around loops of
at least --min-seconds after a warm-up; the best of --rounds is reported, all rounds are recorded.  The loops rotate through several (A, B, C) sets totalling more than the 126 MB
L2, so the operands come from HBM.  TFLOP/s = 2 M N K / time.  torch.matmul writes C in the input type unless this
torch offers torch.mm(..., out_dtype=torch.float32); the line records which.  The GPU name, power limit and maximum SM
clock are read in the same call and written into every line.  ratio_to_torch = torch time / mfa time (> 1: faster).

    python scripts/bench_gemm.py --out profiles/gemm_b200.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 2 ** 20


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True).strip()
        name, power, clock = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:  # report the failure instead of inventing a value
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({exc!r})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,8192")
    ap.add_argument("--dtypes", default="bf16,fp16")
    ap.add_argument("--rounds", type=int, default=3, help="alternating mfa / torch timing rounds per configuration")
    ap.add_argument("--min-seconds", type=float, default=0.15, help="length of one timed loop")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gemm_b200.jsonl"))
    args = ap.parse_args()

    import torch
    import mfa_b200 as mfa
    assert torch.cuda.is_available(), "bench_gemm.py measures the GPU; there is nothing to measure without one"
    P = mfa.GEMMOperandPrecision
    info = gpu_info()
    stream = torch.cuda.current_stream()
    has_out_dtype = True
    rows = []
    for dtype_name in args.dtypes.split(","):
        dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[dtype_name]
        prec = {"bf16": P.BF16, "fp16": P.FP16}[dtype_name]
        for size in (int(s) for s in args.sizes.split(",")):
            M = N = K = size
            flops = 2.0 * M * N * K
            for c_name in ("fp32", dtype_name):
                c_dtype = torch.float32 if c_name == "fp32" else dtype
                set_bytes = (M * K + K * N) * 2 + M * N * c_dtype.itemsize
                sets = max(2, -(-3 * L2_BYTES // set_bytes))
                gen = torch.Generator(device="cuda").manual_seed(size)
                operands = [(torch.randn(M * K, device="cuda", generator=gen).to(dtype),
                             torch.randn(K * N, device="cuda", generator=gen).to(dtype),
                             torch.empty(M * N, device="cuda", dtype=c_dtype)) for _ in range(sets)]
                for tA in (False, True):
                    for tB in (False, True):
                        d = mfa.GEMMDescriptor()
                        d.matrixDimensions = (M, N, K)
                        d.memoryPrecisions = (prec, prec, P.FP32 if c_name == "fp32" else prec)
                        d.transposeState = (tA, tB)
                        kernel = mfa.GEMMKernel.cached(d)
                        consts = mfa.GEMMFunctionConstantValues()
                        d.setFunctionConstants(consts)

                        def views(s):
                            a, b, _ = operands[s]
                            la = a.view(K, M).T if tA else a.view(M, K)
                            lb = b.view(N, K).T if tB else b.view(K, N)
                            return la, lb

                        def run_mfa(s):
                            a, b, c = operands[s]
                            kernel.encode(consts, [a.data_ptr(), b.data_ptr(), c.data_ptr()], stream=stream.cuda_stream)

                        def run_torch(s):
                            nonlocal has_out_dtype
                            la, lb = views(s)
                            if c_dtype == torch.float32 and has_out_dtype:
                                try:
                                    torch.mm(la, lb, out_dtype=torch.float32)
                                    return
                                except (TypeError, RuntimeError):
                                    has_out_dtype = False
                            torch.matmul(la, lb)

                        est = flops / 1.0e15
                        iters = max(8, int(args.min_seconds / est))

                        def timed(fn):
                            for s in range(sets):  # warm-up of every set
                                fn(s)
                            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            start.record()
                            for i in range(iters):
                                fn(i % sets)
                            end.record()
                            end.synchronize()
                            return start.elapsed_time(end) / 1e3 / iters

                        t_mfa, t_torch = [], []
                        for _ in range(args.rounds):
                            t_mfa.append(timed(run_mfa))
                            t_torch.append(timed(run_torch))
                        # correctness of the timed kernel on set 0 against torch in FP32
                        run_mfa(0)
                        la, lb = views(0)
                        ref = torch.matmul(la.float(), lb.float())
                        got = operands[0][2].view(M, N).float()
                        rel = float((got - ref).abs().max() / ref.abs().max())
                        best_mfa, best_torch = min(t_mfa), min(t_torch)
                        row = dict(info, kernel=kernel.sourceName(), dtype=dtype_name, c_dtype=c_name, M=M, N=N, K=K,
                                   transpose=("T" if tA else "N") + ("T" if tB else "N"), iters=iters, operand_sets=sets,
                                   working_set_mb=round(sets * set_bytes / 2 ** 20),
                                   mfa_ms=round(best_mfa * 1e3, 4), torch_ms=round(best_torch * 1e3, 4),
                                   mfa_tflops=round(flops / best_mfa / 1e12, 1),
                                   torch_tflops=round(flops / best_torch / 1e12, 1),
                                   ratio_to_torch=round(best_torch / best_mfa, 3),
                                   mfa_ms_rounds=[round(t * 1e3, 4) for t in t_mfa],
                                   torch_ms_rounds=[round(t * 1e3, 4) for t in t_torch],
                                   torch_c_dtype=("fp32" if c_dtype == torch.float32 and has_out_dtype else dtype_name),
                                   max_rel_err_vs_torch_fp32=rel, unix_time=int(time.time()))
                        print(json.dumps(row), flush=True)
                        rows.append(row)
                del operands
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
