#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on B200: giga-FMA-instructions/s (and TFLOP/s) of the
FlashAttention forward at N=4096, D=128, bf16 in / fp32 out.

One "step" = one pass of the hot path over one batch of synthetic input: H independent single-head
(N=4096, D=128) problems per GPU, one kernel launch (the reference is single-head; independent heads
are the only thing that scales, SURVEY.md section 8(e)).  Work model is the reference's:
(2D+5)*N^2 FMA-instructions per head forward (README.md:108-124; SquareAttentionTest.swift:742-756);
TFLOP/s counts the two GEMMs only, 4*N^2*D per head.

    python bench.py --gpus 1 --steps 50 --warmup 5            # our arm
    python bench.py --gpus 1 --steps 50 --warmup 5 --dump-outputs DIR   # ... and keep a sample of O and L to compare
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1   # the reference's CPU path (oracle port)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  Inputs
for one step (Q,K,V = 192 MiB at H=64) exceed the 126 MB L2 and two buffer sets alternate between steps.
`e2e` goes through the C ABI's host-buffer entry point (mfa_attention_run_host: pinned host Q,K,V -> device,
kernel, O and L -> host) inside the timed region; the host buffers come from mfa_host_alloc (page-locked, on the
GPU's NUMA node) and every rank pins itself to its GPU's socket first.

Further legs on the same JSON line (none of them replaces `value`):
  sustained  the same step looped for >= 2 s: the power-capped regime, fraction against bf16_tflops_sustained
  config5    BASELINE.json configs[4] as written: 64 x 32 = 2048 independent (N=4096, D=128) problems block-partitioned
             over the ranks; data starts on rank 0 (NCCL send/recv scatter), O and L end on rank 0 (gather); kernel
             time and the scatter / gather times are reported separately (SURVEY.md section 8(d)/(e))
  single_head one problem per call (split-KV across the SMs, merged inside the kernel)
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_SEQ, D_HEAD = 4096, 128
FMA_PER_HEAD = (2 * D_HEAD + 5) * N_SEQ * N_SEQ          # reference's forward work model
FLOP_PER_HEAD = 4 * N_SEQ * N_SEQ * D_HEAD               # two GEMMs
METRIC = "giga-FMA-instr/sec forward attn N=4096 D=128 bf16"
UNIT = "GINSTRS"
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture
# (profiles/), for the default H; None until a capture exists.
NCU_TRAFFIC_BYTES_PER_LAUNCH = 298728960  # profiles/r2_fwd_ncu_summary.csv: 201.77 MB read + 96.96 MB written
NCU_TRAFFIC_SOURCE = "profiles/r2_fwd_ncu_summary.csv (ncu --set full, one 64-head launch of this kernel; not re-measured in this run)"
# --dump-outputs keeps this many (head, row) rows of O and L: 32 MiB of O at D=128, whatever --heads is
DUMP_ROWS, DUMP_SEED = 65536, 0


def dump_outputs(directory, o, lse):
    """Write a fixed, seeded sample of the rows of O [H, N, D] and L [H, N] as float32 .npy files.  The sample depends
    only on H and N, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    rows = o.shape[0] * o.shape[1]
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(rows, size=min(rows, DUMP_ROWS), replace=False))
    index = torch.from_numpy(pick).to(o.device)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "O.npy"), o.reshape(rows, -1).index_select(0, index).float().cpu().numpy())
    np.save(os.path.join(directory, "L.npy"), lse.reshape(rows).index_select(0, index).float().cpu().numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            peaks = json.load(f)
        return float(peaks["bf16_tflops"]), float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])), "measured"
    return 1590.0, 1400.0, "fallback"   # /opt/skills/guides/B200_PROFILING.md


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, device_index, period_s=0.0005):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # NVML missing: report that instead of inventing numbers
            self._nvml, self._error = None, repr(exc)
        self.period = period_s

    def _loop(self):
        nv = self._nvml
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self._nvml:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread:
            self._thread.join()
            # one more reading right at the end of the timed region (the kernels have only just drained): short runs
            # otherwise end up with a single sample
            try:
                self.samples.append(self._nvml.nvmlDeviceGetClockInfo(self._handle, self._nvml.NVML_CLOCK_SM))
            except Exception:
                pass

    def summary(self):
        if not self._nvml:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": self._error}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def host_tensor(mfa, shape, dtype, device, upload=False):
    """A torch view of a page-locked buffer from mfa_host_alloc (NUMA-local to `device`); returns (tensor, address)."""
    import ctypes
    import torch
    nbytes = 1
    for n in shape:
        nbytes *= int(n)
    nbytes *= torch.empty((), dtype=dtype).element_size()
    addr = mfa.hostAlloc(nbytes, device, upload=upload)
    raw = (ctypes.c_uint8 * nbytes).from_address(addr)
    return torch.frombuffer(raw, dtype=torch.uint8).view(dtype).reshape(tuple(shape)), addr


def run_config5(args, mfa, torch, dist, rank, world, stream, heads_per_launch):
    """BASELINE.json configs[4]: `total` independent (N=4096, D=128) problems, contiguous block partition over the
    ranks (sharding.head_partition).  All inputs start on rank 0 and reach the shards through NCCL send/recv, every
    rank runs the same single-GPU kernel over its shard in launches of `heads_per_launch`, O and L are gathered back to
    rank 0.  Scatter, kernels and gather are timed separately with CUDA events (max over ranks)."""
    from mfa_b200.sharding import head_partition, scatter_heads, gather_heads
    Op = mfa.AttentionOperand
    total = args.config5_heads
    start_head, count = head_partition(total, world, rank)
    dev = torch.device("cuda", torch.cuda.current_device())
    full = {}
    if rank == 0:
        gen = torch.Generator(device="cuda").manual_seed(77)
        for op in (Op.Q, Op.K, Op.V):
            full[op] = torch.empty(total, N_SEQ, D_HEAD, device="cuda", dtype=torch.bfloat16)
            for h0 in range(0, total, 64):   # generated in slices: the FP32 staging of randn stays small
                n = min(64, total - h0)
                full[op][h0:h0 + n] = torch.randn(n, N_SEQ, D_HEAD, device="cuda", generator=gen).to(torch.bfloat16)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        a.record(stream)
        out = fn()
        b.record(stream)
        sync()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return out, ms

    if world > 1:   # open the NCCL point-to-point connections outside the timed region
        warm = torch.zeros(world, 1024, device="cuda") if rank == 0 else None
        piece = scatter_heads(warm, world, (1024,), torch.float32, dev)
        gather_heads(piece, world)   # (the peer -> rank 0 direction is a separate set of connections)

    if world > 1:
        shards, scatter_ms = timed(lambda: {op: scatter_heads(full.get(op), total, (N_SEQ, D_HEAD), torch.bfloat16, dev)
                                            for op in (Op.Q, Op.K, Op.V)})
    else:   # one rank owns everything: nothing to scatter
        shards, scatter_ms = {op: full[op] for op in (Op.Q, Op.K, Op.V)}, 0.0
    scatter_bytes = 3 * (total - head_partition(total, world, 0)[1]) * N_SEQ * D_HEAD * 2

    o = torch.empty(count, N_SEQ, D_HEAD, device="cuda", dtype=torch.float32)
    lse = torch.empty(count, N_SEQ, device="cuda", dtype=torch.float32)
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    desc.matrixDimensions = (N_SEQ, N_SEQ, D_HEAD)
    desc.transposeState = (False, False, False, False)
    launches = []
    for h0 in range(0, count, heads_per_launch):
        n = min(heads_per_launch, count - h0)
        desc.batchCount = n
        c = mfa.FunctionConstantValues()
        desc.setFunctionConstants(c)
        ptrs = {Op.Q: shards[Op.Q][h0:].data_ptr(), Op.K: shards[Op.K][h0:].data_ptr(),
                Op.V: shards[Op.V][h0:].data_ptr(), Op.O: o[h0:].data_ptr(), Op.L: lse[h0:].data_ptr()}
        launches.append((c, ptrs))
    kernel = mfa.AttentionKernel.cached(desc, mfa.AttentionKernelType.forward)

    def compute():
        for c, ptrs in launches:
            kernel.encode(c, ptrs, stream.cuda_stream)

    compute()   # warm (first touch of O / L)
    _, kernel_ms = timed(compute)
    if world > 1:
        # destination on rank 0 allocated (and touched) outside the timed region: the transfer is what is measured
        out_o = torch.zeros(total, N_SEQ, D_HEAD, device="cuda", dtype=torch.float32) if rank == 0 else None
        out_l = torch.zeros(total, N_SEQ, device="cuda", dtype=torch.float32) if rank == 0 else None
        (full_o, full_l), gather_ms = timed(lambda: (gather_heads(o, total, out=out_o), gather_heads(lse, total, out=out_l)))
    else:
        (full_o, full_l), gather_ms = (o, lse), 0.0
    gather_bytes = (total - head_partition(total, world, 0)[1]) * (N_SEQ * D_HEAD + N_SEQ) * 4
    ok = None
    if rank == 0:
        # the gathered result is the per-shard result: spot-check a head that travelled (the last one) through the
        # softmax identity rowsum(P) = 1  <=>  O with V := 1 ... not available here, so check finiteness and L's range
        last = full_o[total - 1]
        ok = bool(torch.isfinite(last).all().item()) and bool(torch.isfinite(full_l[total - 1]).all().item())
    work = FMA_PER_HEAD * total
    return {
        "workload": f"{total} independent (N=4096, D=128) bf16 problems = batch 64 x heads 32, block-partitioned over "
                    f"{world} GPU(s): {count} on this rank, launches of {heads_per_launch}",
        "kernel_ms": kernel_ms, "kernel_ginstrs": work / kernel_ms / 1e6,
        "kernel_tflops": FLOP_PER_HEAD * total / kernel_ms / 1e9,
        "scatter_ms": scatter_ms, "gather_ms": gather_ms,
        "scatter_bytes": scatter_bytes, "gather_bytes": gather_bytes,
        "scatter_gbs": (scatter_bytes / scatter_ms / 1e6) if world > 1 and scatter_ms > 0 else None,
        "gather_gbs": (gather_bytes / gather_ms / 1e6) if world > 1 and gather_ms > 0 else None,
        "with_scatter_gather_ms": scatter_ms + kernel_ms + gather_ms,
        "with_scatter_gather_ginstrs": work / (scatter_ms + kernel_ms + gather_ms) / 1e6,
        "comm": {"backend": dist.get_backend() if world > 1 else None, "nranks": world,
                 "p2p_messages": 5 * (world - 1),
                 "pattern": "rank 0 -> ranks: ncclSend/ncclRecv of Q, K, V shards; ranks -> rank 0: O, L shards"},
        "gathered_result_finite": ok,
    }


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  The reference (Swift) cannot be
    built here, so this is the C port of its `Network` oracle (oracle/network_oracle.c), row-parallel over all
    host threads.  Each step is a bounded sample of the workload: ONE head (N=4096, D=128) forward."""
    if rank != 0:
        return
    import oracle
    # every host core this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle's num_threads clause
    # takes the explicit count, so the CPU arm is not throttled by the launcher)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    net = oracle.Network(N_SEQ, N_SEQ, D_HEAD, seed=0, threads=threads)
    for _ in range(args.warmup):
        net.inferenceAttention()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        net.inferenceAttention()
    dt = time.perf_counter() - t0
    value = FMA_PER_HEAD * args.steps / dt / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "tflops": FLOP_PER_HEAD * args.steps / dt / 1e12,
        "config": {"workload": "forward attention N=4096 D=128, 1 head per step (bounded sample of the "
                               "H-head step), FP32, reference CPU path = C port of Tests/.../Network.swift",
                   "seq_len": N_SEQ, "head_dim": D_HEAD, "heads_per_step": 1},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "1 head (N=4096, D=128) forward per step, rows split over all host threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--heads", type=int, default=64, help="independent single-head problems per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--config5-heads", type=int, default=2048, help="batch 64 x heads 32 of BASELINE.json configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's O and L of the last timed step to DIR/O.npy and DIR/L.npy "
                         f"(float32; a fixed seeded sample of at most {DUMP_ROWS} of the heads x N rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import mfa_b200 as mfa   # raises if libmfa_b200.so is missing: there is no fallback path

    assert torch.cuda.is_available(), "bench.py (our arm) needs a B200"
    torch.cuda.set_device(local_rank)
    # this rank's host threads (and everything it allocates from here on: pinned staging buffers, NCCL proxies) stay on
    # the socket its GPU hangs off -- the H2D / D2H copies of the e2e leg never cross the inter-socket link
    numa_node = mfa.bindThreadToDevice(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    H = args.heads

    # ---- descriptor -> kernel, exactly as a client of the reference API would -------------------
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = True
    desc.lowPrecisionIntermediates = False
    desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    desc.matrixDimensions = (N_SEQ, N_SEQ, D_HEAD)
    desc.transposeState = (False, False, False, False)
    desc.batchCount = H
    kernel_desc = desc.kernelDescriptor(mfa.AttentionKernelType.forward)
    assert kernel_desc.backend == mfa.Backend.tcgen05
    kernel = mfa.AttentionKernel(kernel_desc)
    constants = mfa.FunctionConstantValues()
    desc.setFunctionConstants(constants)
    launches_per_step = kernel.launchCount(constants)
    Op = mfa.AttentionOperand

    # ---- synthetic inputs, resident in HBM; two sets so consecutive steps never share lines -----
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    sets = []
    for _ in range(2):
        q, k, v = (torch.randn(H, N_SEQ, D_HEAD, device="cuda", dtype=torch.float32, generator=gen).to(torch.bfloat16)
                   for _ in range(3))
        o = torch.empty(H, N_SEQ, D_HEAD, device="cuda", dtype=torch.float32)
        lse = torch.empty(H, N_SEQ, device="cuda", dtype=torch.float32)
        sets.append({Op.Q: q, Op.K: k, Op.V: v, Op.O: o, Op.L: lse})
    stream = torch.cuda.current_stream()

    def step(i):
        bufs = sets[i & 1]
        kernel.encode(constants, {op: t.data_ptr() for op, t in bufs.items()}, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()

    # ---- `value`: device-timed, inputs resident ------------------------------------------------
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    ids = [x for x in visible.split(",") if x.strip().isdigit()]
    sampler = ClockSampler(int(ids[local_rank]) if local_rank < len(ids) else local_rank)
    with sampler:
        barrier()
        start.record(stream)
        for i in range(args.steps):
            step(i)
        stop.record(stream)
        barrier()
    elapsed_ms = start.elapsed_time(stop)
    if world > 1:
        t = torch.tensor([elapsed_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    total_heads = H * world
    value = FMA_PER_HEAD * total_heads / (ms_per_step * 1e-3) / 1e9
    tflops = FLOP_PER_HEAD * total_heads / (ms_per_step * 1e-3) / 1e12
    if args.dump_outputs and rank == 0:   # before the legs below launch on the same buffers again
        last = sets[(args.steps - 1) & 1]
        dump_outputs(args.dump_outputs, last[Op.O], last[Op.L])

    # ---- `e2e`: host buffers through mfa_attention_run_host ------------------------------------
    e2e = None
    if not args.no_e2e:
        host, host_addr = {}, {}
        for op, t in sets[0].items():
            host[op], host_addr[op] = host_tensor(mfa, t.shape, t.dtype, torch.cuda.current_device(),
                                                  upload=op in (Op.Q, Op.K, Op.V) and not os.environ.get("MFA_B200_BENCH_NO_WC"))
            # (write-combined upload buffers: the host only writes them; MFA_B200_BENCH_NO_WC=1 is the A/B switch)
            if op in (Op.Q, Op.K, Op.V):
                host[op].copy_(t.cpu())
        host_ptrs = dict(host_addr)
        fwd = [mfa.AttentionKernelType.forward]
        e2e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            desc.runHost(fwd, host_ptrs, device=torch.cuda.current_device())
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            desc.runHost(fwd, host_ptrs, device=torch.cuda.current_device())   # synchronous: returns after D2H
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        h2d = sum(host[op].numel() * host[op].element_size() for op in (Op.Q, Op.K, Op.V))
        d2h = sum(host[op].numel() * host[op].element_size() for op in (Op.O, Op.L))
        e2e = {"value": FMA_PER_HEAD * total_heads * e2e_steps / dt / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
               "ms_per_step": dt / e2e_steps * 1e3,
               "api": "mfa_attention_run_host (pinned host Q,K,V -> device, kernel, O,L -> host)",
               "host_buffers": "mfa_host_alloc (O, L) / mfa_host_alloc_upload (Q, K, V: write-combined): cudaHostAlloc(portable) "
                               "first-touched on the GPU's NUMA node",
               "numa_node": numa_node}
        # spot-check that the e2e path produced the same O as the device path.  The host path works through the batch in
        # chunks of a few heads, for which the library may split the key axis across SMs and merge; each split rounds
        # P to BF16 against its own running maximum, so the two paths agree to the kernel's accuracy (relative RMS
        # 2e-3, tests/test_tcgen05_forward.py), not bit for bit.
        step(0)
        torch.cuda.synchronize()
        for sl in ((0, slice(0, 64)), (H - 1, slice(N_SEQ - 64, N_SEQ))):
            got, want = host[Op.O][sl].float(), sets[0][Op.O][sl].cpu().float()
            rel = float((got - want).norm() / want.norm())
            assert rel < 4e-3, f"e2e != device path (relative RMS {rel:.2e})"
        del host
        for addr in host_addr.values():
            mfa.hostFree(addr)

    # ---- literal single-head latency (BASELINE.json configs[1] as written): one (N=4096, D=128) problem per launch;
    #      too few tiles to fill 148 SMs, so the library splits the key axis across SMs and merges (split-KV) --------
    single_head = None
    if rank == 0:
        d1 = mfa.AttentionDescriptor()
        d1.lowPrecisionInputs = True
        d1.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
        d1.matrixDimensions = (N_SEQ, N_SEQ, D_HEAD)
        d1.transposeState = (False, False, False, False)
        k1 = mfa.AttentionKernel(d1.kernelDescriptor(mfa.AttentionKernelType.forward))
        c1 = mfa.FunctionConstantValues()
        d1.setFunctionConstants(c1)
        ptrs = {op: t[0].data_ptr() for op, t in sets[0].items()}
        for _ in range(5):
            k1.encode(c1, ptrs, stream.cuda_stream)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 50
        a.record(stream)
        for _ in range(reps):
            k1.encode(c1, ptrs, stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        ms1 = a.elapsed_time(b) / reps
        single_head = {"ms_per_launch": ms1, "ginstrs": FMA_PER_HEAD / ms1 / 1e6, "tflops": FLOP_PER_HEAD / ms1 / 1e9,
                       "launches_per_call": k1.launchCount(c1),
                       "note": "one head per call, 50 back-to-back calls, inputs L2-resident (5 MB problem)"}

    # ---- sustained regime: the same step looped for >= 2 s (power-capped clocks), every rank in lock step ----------
    sustained = None
    if not args.no_sustained:
        reps = max(1, int(args.sustained_seconds * 1e3 / ms_per_step))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sus_sampler = ClockSampler(int(ids[local_rank]) if local_rank < len(ids) else local_rank, period_s=0.01)
        with sus_sampler:
            barrier()
            a.record(stream)
            for i in range(reps):
                step(i)
            b.record(stream)
            barrier()
        sus_ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([sus_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sus_ms = float(t.item())
        sustained = {"seconds": sus_ms / 1e3, "steps": reps, "ms_per_step": sus_ms / reps,
                     "tflops_per_gpu": FLOP_PER_HEAD * H * reps / sus_ms / 1e9,
                     "ginstrs": FMA_PER_HEAD * total_heads * reps / sus_ms / 1e6, "clocks": sus_sampler.summary()}

    # ---- BASELINE.json configs[4] as written: 2048 problems over the ranks, NCCL scatter / gather timed apart --------
    config5 = None
    if not args.no_config5:
        config5 = run_config5(args, mfa, torch, dist, rank, world, stream, H)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel -------------------------------------------------
    peak_burst, peak_sustained, peak_kind = measured_peaks()
    per_gpu_tflops = FLOP_PER_HEAD * H / (ms_per_step * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "achieved": per_gpu_tflops, "peak": peak_burst, "unit": "TFLOP/s",
        "frac": per_gpu_tflops / peak_burst, "traffic": NCU_TRAFFIC_BYTES_PER_LAUNCH,
        "peak_kind": f"{peak_kind} cuBLAS bf16 burst (MEASURED_PEAKS.json)" if peak_kind == "measured"
                     else "fallback 1590 TF/s (B200_PROFILING.md)",
        "kernel": kernel.sourceName(), "flops_per_launch": FLOP_PER_HEAD * H,
        "kernel_ms": ms_per_step, "algorithmic_bytes_per_launch": H * (3 * N_SEQ * D_HEAD * 2 + N_SEQ * D_HEAD * 4 + N_SEQ * 4),
        "traffic_source": NCU_TRAFFIC_SOURCE,
    }
    if sustained is not None:
        # like for like: seconds of back-to-back launches against the seconds-long cuBLAS figure
        sustained["peak"] = peak_sustained
        sustained["frac_of_sustained_peak"] = sustained["tflops_per_gpu"] / peak_sustained

    # ---- CPU baseline: the oracle port, single thread "as written", on a bounded sample ----------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        import oracle
        net = oracle.Network(N_SEQ, N_SEQ, D_HEAD, seed=0, threads=1)
        t0 = time.perf_counter()
        net.inferenceAttention()
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": FMA_PER_HEAD / dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": f"1 of the {H} heads of one step (N=4096, D=128), single thread, "
                                  f"loop order of Network.inferenceAttention; {dt:.1f} s"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "tflops": tflops,
        "config": {"workload": f"forward attention, {H} independent single-head problems per GPU per step, "
                               "N=4096 D=128, bf16 Q/K/V, fp32 O and L (BASELINE.json configs[1] x heads)",
                   "seq_len": N_SEQ, "head_dim": D_HEAD, "heads_per_gpu_per_step": H,
                   "parallelism": f"heads sharded over {world} GPU(s), no data-path collective",
                   "l2": "inputs per step (192 MiB at H=64) exceed the 126 MB L2; two buffer sets alternate"},
        "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": args.steps * launches_per_step,
        "roofline": roofline, "cpu_baseline": cpu_baseline, "single_head": single_head,
        "sustained": sustained, "config5": config5, "numa_node": numa_node,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
