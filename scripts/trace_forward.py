"""Pipeline timeline of the tcgen05 forward kernel (debug instantiation with clock64() probes).
Usage on the GPU box:  python scripts/trace_forward.py [R] [heads]  -> prints per-iteration cycle deltas."""
import ctypes
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mfa_b200 as mfa  # noqa: E402

R = int(sys.argv[1]) if len(sys.argv) > 1 else 256
H = int(sys.argv[2]) if len(sys.argv) > 2 else 1
C, D = 4096, 128

desc = mfa.AttentionDescriptor()
desc.lowPrecisionInputs = True
desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
desc.matrixDimensions = (R, C, D)
desc.transposeState = (False,) * 4
desc.batchCount = H
kernel = mfa.AttentionKernel(desc.kernelDescriptor(mfa.AttentionKernelType.forward))
constants = mfa.FunctionConstantValues()
desc.setFunctionConstants(constants)

q = torch.randn(H, R, D, device="cuda").to(torch.bfloat16)
k = torch.randn(H, C, D, device="cuda").to(torch.bfloat16)
v = torch.randn(H, C, D, device="cuda").to(torch.bfloat16)
o = torch.empty(H, R, D, device="cuda")
lse = torch.empty(H, R, device="cuda")
trace = torch.zeros(8 * 64 * 8, dtype=torch.int64, device="cuda")

lib = mfa._lib
lib.mfa_debug_forward_trace.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p]
arr = (ctypes.c_void_p * 10)()
for slot, t in ((0, q), (1, k), (2, v), (3, o), (4, lse)):
    arr[slot] = t.data_ptr()
for _ in range(3):
    st = lib.mfa_debug_forward_trace(kernel._handle, ctypes.byref(constants._c), ctypes.byref(arr), None,
                                     ctypes.c_void_p(trace.data_ptr()))
    assert st == 0, lib.mfa_last_error()
    torch.cuda.synchronize()
t = trace.cpu().numpy().reshape(8, 64, 8)
nb = C // 128
t0 = t[2, 0, 0]
print(f"R={R} H={H}: cycles relative to MMA warp's first V wait; softmax slots: 0 S ready, 1 S in regs, 2 max done, "
      "3 P computed, 4 arrived; mma slots: 0 V ready, 1 p0 ready, 2 p1(tile 0) ready [then waits K(j+1)], 3 S0 issued, 4 p1 ready, 5 PV1 issued, 6 S1 issued")
for j in range(min(nb, 12)):
    a = (t[0, j, :5] - t0).tolist()
    b = (t[1, j, :5] - t0).tolist()
    m = (t[2, j, :7] - t0).tolist()
    pr = (t[3, j, :3] - t0).tolist()
    print(f"j={j:2d} sm0 {a}  sm1 {b}  mma {m}  tma[wait k_empty, K issue, V issue] {pr}")
per_iter = np.diff(t[2, 2:nb - 1, 1]).mean()
sm = t[0, 2:nb - 1]
print(f"steady-state period per key block: {per_iter:.0f} cycles (ideal 2048 tensor / 2048 MUFU)")
print(f"softmax tile0: wait-for-S->S-in-regs {np.mean(sm[:,1]-sm[:,0]):.0f}, max {np.mean(sm[:,2]-sm[:,1]):.0f}, "
      f"exp+pack+st {np.mean(sm[:,3]-sm[:,2]):.0f}, wait_st+arrive {np.mean(sm[:,4]-sm[:,3]):.0f}, "
      f"arrive->next S ready {np.mean(sm[1:,0]-sm[:-1,4]):.0f}")
mm = t[2, 2:nb - 1]
print(f"mma: p0 ready->PV0+S0 issued {np.mean(mm[:,3]-mm[:,1]):.0f}; S0 issued->p1 ready {np.mean(mm[:,4]-mm[:,3]):.0f}; "
      f"p1 ready->issued {np.mean(mm[:,6]-mm[:,4]):.0f}; S1 issued -> next p0 ready {np.mean(mm[1:,1]-mm[:-1,6]):.0f}")
# MMA latency: time from S0 issue (slot 3 of iter j) to softmax0 seeing S ready (slot 0 of iter j+1)
print(f"S0 issue -> softmax0 sees S(j+1): {np.mean(t[0,3:nb-1,0]-t[2,2:nb-2,3]):.0f} cycles; "
      f"softmax0 arrive(j) -> mma sees p0(j): {np.mean(t[2,2:nb-1,1]-t[0,2:nb-1,4]):.0f}")

# ---- item-level timeline of CTA 0 (persistent kernel): roles 4/5 = softmax tile 0/1, role 6 = MMA warp
items = int((t[4, :, 0] != 0).sum())
base = t[6, 0, 0]
print(f"items processed by CTA 0: {items}; per item (cycles from the MMA warp's first prologue):")
for it in range(min(items, 8)):
    a = (t[4, it, :4] - base).tolist(); b2 = (t[5, it, :4] - base).tolist(); mm2 = (t[6, it, :3] - base).tolist()
    print(f" it={it} tile0 [start, loop end, O ready, epilogue end] {a}  tile1 {b2}  mma [prologue, S(0) issued, loop end] {mm2}")
if items > 2:
    per_item = np.diff(t[4, 1:items, 0]).mean()
    print(f"cycles per item {per_item:.0f}; loop {np.mean(t[4,1:items,1]-t[4,1:items,0]):.0f}; wait O {np.mean(t[4,1:items,2]-t[4,1:items,1]):.0f}; "
          f"epilogue {np.mean(t[4,1:items,3]-t[4,1:items,2]):.0f}; epilogue end -> next start {np.mean(t[4,2:items,0]-t[4,1:items-1,3]):.0f}")
    first = t[0, 0:4, 4] - t[0, 0:4, 0]
    print("first four blocks of the last item, S ready -> P arrived (tile 0):", first.tolist())
