"""Host-side logic of the GEMM half of the C ABI (no GPU): GEMMDescriptor.setFunctionConstants, the kernel-descriptor
heuristic, GEMMKernel validation and geometry, the pipeline cache, and the C++ mirror.  Mirrors what the reference's
Swift GEMM types do on the CPU (Sources/FlashAttention/GEMM/)."""
import itertools
import os
import subprocess

import pytest

import mfa_b200 as mfa
from mfa_b200 import GEMMOperandPrecision as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRANSPOSES = [(False, False), (False, True), (True, False), (True, True)]


def make(M=100, N=200, K=300, precisions=(P.FP32, P.FP32, P.FP32), transpose=(False, False), leading=None,
         load_previous=False, batch=1):
    d = mfa.GEMMDescriptor()
    d.matrixDimensions = (M, N, K)
    d.memoryPrecisions = precisions
    d.transposeState = transpose
    d.leadingDimensions = leading
    d.loadPreviousC = load_previous
    d.batchDimension = batch
    return d


def constants(d):
    c = mfa.GEMMFunctionConstantValues()
    d.setFunctionConstants(c)
    return c


def test_default_leading_dimensions_follow_choose_leading_dimension():
    """GEMMDescriptor.swift:340-373: transposed -> untransposed rows, else untransposed columns; C is never transposed."""
    for (tA, tB), expected in zip(TRANSPOSES, [(300, 200, 200), (300, 300, 200), (100, 200, 200), (100, 300, 200)]):
        c = constants(make(transpose=(tA, tB)))
        assert c.leadingDimensions == expected
        assert c.matrixDimensions == (100, 200, 300) and not c.loadPreviousC and c.batchCount == 1
    c = constants(make(leading=(301, 260, 999), load_previous=True, batch=4))
    assert c.leadingDimensions == (301, 260, 999) and c.loadPreviousC and c.batchCount == 4


@pytest.mark.parametrize("leading", [(299, 200, 200), (300, 199, 200), (300, 200, 199)])
def test_leading_dimension_too_small_is_an_error(leading):
    with pytest.raises(mfa.MFAError, match="Leading block dimension was too small."):
        constants(make(leading=leading))
    # transposed A: the minimum is M (100), so 150 < K is fine there
    constants(make(transpose=(True, False), leading=(150, 200, 200)))


def test_incomplete_descriptors_carry_the_reference_message():
    for missing in ("matrixDimensions", "memoryPrecisions", "transposeState"):
        d = make()
        setattr(d, missing, None)
        with pytest.raises(mfa.MFAError, match="Descriptor was incomplete.") as err:   # GEMMDescriptor.swift:107-111
            mfa.GEMMKernelDescriptor(d)
        assert err.value.status == -1
        with pytest.raises(mfa.MFAError, match="Descriptor was incomplete."):
            mfa.GEMMKernel.cached(d)
    d = make()
    d.transposeState = None
    with pytest.raises(mfa.MFAError, match="Descriptor was incomplete."):             # :328-331
        constants(d)
    with pytest.raises(mfa.MFAError, match="Descriptor was incomplete."):             # GEMMKernel.swift:27-34
        mfa.GEMMKernel(mfa.GEMMKernelDescriptor())
    kd = mfa.GEMMKernelDescriptor(make())
    kd.preferAsyncStore = None
    with pytest.raises(mfa.MFAError, match="Descriptor was incomplete."):
        mfa.GEMMKernel(kd)


@pytest.mark.parametrize("transpose", TRANSPOSES)
def test_backend_over_the_whole_precision_grid(transpose):
    """tcgen05 exactly when A and B are both FP16 or both BF16 (any C); SIMT FP32 otherwise."""
    for a, b, c in itertools.product(P, P, P):
        kd = mfa.GEMMKernelDescriptor(make(precisions=(a, b, c), transpose=transpose))
        tc = a == b and a != P.FP32
        assert kd.backend == (mfa.Backend.tcgen05 if tc else mfa.Backend.simtFP32), (a, b, c)
        assert kd.memoryPrecisions == (a, b, c)
        assert kd.registerPrecisions == (a, b, P.FP32)        # the accumulator is FP32 in TMEM or in registers
        assert kd.transposeState == transpose
        assert kd.preferAsyncLoad == tc and kd.preferAsyncStore is False
        k = mfa.GEMMKernel(kd)
        name = k.sourceName()
        assert name.startswith("gemm_tcgen05<" if tc else "gemm_simt_fp32<")
        assert name.endswith(("T" if transpose[0] else "N") + ("T" if transpose[1] else "N") + ">")


@pytest.mark.parametrize("transpose", TRANSPOSES)
def test_kernel_geometry(transpose):
    tA, tB = transpose
    tc = mfa.GEMMKernelDescriptor(make(precisions=(P.BF16, P.BF16, P.FP32), transpose=transpose))
    assert tc.blockDimensions == (128, 256, 64) and tc.splits == (4, 1)
    assert tc.leadingBlockDimensions == (128 if tA else 64, 64 if tB else 256, 256)
    k = mfa.GEMMKernel(tc)
    assert k.blockDimensions == (128, 256, 64) and k.threadgroupSize == 192
    assert 4 * 48 * 1024 < k.threadgroupMemoryAllocation <= 232448        # one CTA per SM: it owns all of TMEM
    assert 2 * k.threadgroupMemoryAllocation > 233472
    simt = mfa.GEMMKernelDescriptor(make(transpose=transpose))
    assert simt.blockDimensions == (64, 64, 16) and simt.splits == (2, 4)
    assert simt.leadingBlockDimensions == (64 if tA else 16, 16 if tB else 64, 64)
    s = mfa.GEMMKernel(simt)
    assert s.threadgroupSize == 32 * 2 * 4 and 0 < s.threadgroupMemoryAllocation <= 48 * 1024

    # gridSize: output tiles, AdversarialShapeTest.swift:155-158, times the batch
    for (M, N, batch) in ((1, 1, 1), (128, 256, 1), (129, 257, 1), (1000, 600, 3)):
        c = constants(make(M=M, N=N, batch=batch, transpose=transpose))
        assert k.gridSize(c) == -(-M // 128) * -(-N // 256) * batch
        assert s.gridSize(c) == -(-M // 64) * -(-N // 64) * batch


def test_launch_count_counts_the_staging_copies():
    def count(precisions, transpose, leading):
        d = make(M=64, N=64, K=64, precisions=precisions, transpose=transpose, leading=leading)
        return mfa.GEMMKernel.cached(d).launchCount(constants(d))
    bf16 = (P.BF16, P.BF16, P.FP32)
    for t in TRANSPOSES:
        assert count(bf16, t, (64, 64, 64)) == 1
        assert count(bf16, t, (65, 64, 64)) == 2
        assert count(bf16, t, (64, 70, 64)) == 2
        assert count(bf16, t, (67, 71, 64)) == 3
        assert count(bf16, t, (64, 64, 65)) == 1         # C is stored with plain st.global: any ldc
        assert count((P.FP32, P.FP32, P.FP32), t, (67, 71, 65)) == 1   # the SIMT kernel reads any layout in place


def test_register_precision_truth_table():
    """GEMMKernel.swift:46-103, with the reference's messages."""
    base = make(precisions=(P.FP16, P.FP16, P.FP16))
    for operand, index in (("A", 0), ("B", 1)):
        kd = mfa.GEMMKernelDescriptor(base)
        reg = list(kd.registerPrecisions)
        reg[index] = P.BF16                                             # FP16 memory -> BF16 register
        kd.registerPrecisions = tuple(reg)
        with pytest.raises(mfa.MFAError, match=f"Operand {operand} had an invalid register precision.") as err:
            mfa.GEMMKernel(kd)
        assert err.value.status == -4
    kd = mfa.GEMMKernelDescriptor(make())                               # FP32 memory -> FP16 register
    kd.registerPrecisions = (P.FP32, P.FP32, P.FP16)
    with pytest.raises(mfa.MFAError, match="Operand C had an invalid register precision."):
        mfa.GEMMKernel(kd)
    kd = mfa.GEMMKernelDescriptor(make(precisions=(P.BF16, P.BF16, P.BF16)))
    kd.registerPrecisions = (P.BF16, P.BF16, P.BF16)
    with pytest.raises(mfa.MFAError, match="BF16 cannot be used as the register precision for C."):
        mfa.GEMMKernel(kd)
    # legal in the reference: an FP16 accumulator for FP16 C (the kernel still accumulates in FP32)
    kd = mfa.GEMMKernelDescriptor(base)
    kd.registerPrecisions = (P.FP16, P.FP16, P.FP16)
    assert "tcgen05" in mfa.GEMMKernel(kd).sourceName()
    kd.registerPrecisions = (P.FP32, P.FP32, P.FP32)                    # widened inputs: also legal
    mfa.GEMMKernel(kd)


def test_edited_kernel_descriptors_outside_compiled_kernels_are_rejected():
    kd = mfa.GEMMKernelDescriptor(make(precisions=(P.FP16, P.FP16, P.FP32)))
    kd.blockDimensions = (48, 48, 32)                                   # an Apple tile shape
    with pytest.raises(mfa.MFAError, match="no compiled sm_100a kernel"):
        mfa.GEMMKernel(kd)
    kd = mfa.GEMMKernelDescriptor(make(precisions=(P.FP16, P.FP16, P.FP32)))
    kd.leadingBlockDimensions = (32, 256, 256)
    with pytest.raises(mfa.MFAError, match="Leading block dimension was too small."):
        mfa.GEMMKernel(kd)
    kd.leadingBlockDimensions = None                                    # optional: defaults to the compiled layout
    mfa.GEMMKernel(kd)
    kd = mfa.GEMMKernelDescriptor(make(precisions=(P.FP16, P.BF16, P.FP32)))
    assert kd.backend == mfa.Backend.simtFP32
    kd.backend = mfa.Backend.tcgen05
    kd.blockDimensions = (128, 256, 64)
    with pytest.raises(mfa.MFAError, match="MFA_BACKEND_TCGEN05 needs A and B"):
        mfa.GEMMKernel(kd)


def test_pipeline_cache_keys_on_precisions_and_transposes():
    """GEMMDescriptor+PipelineCache.swift:16-36: M, N, K, the leading dimensions, loadPreviousC and the batch are launch
    constants; precisions and transposes select the kernel."""
    before = mfa.GEMMKernel.cacheSize()
    prec = (P.FP16, P.FP16, P.BF16)
    a = mfa.GEMMKernel.cached(make(precisions=prec, transpose=(True, True)))
    b = mfa.GEMMKernel.cached(make(7, 9, 11, precisions=prec, transpose=(True, True), leading=(40, 50, 60),
                                   load_previous=True, batch=3))
    assert a._handle.value == b._handle.value and mfa.GEMMKernel.cacheSize() == before + 1
    mfa.GEMMKernel.register(make(5000, 1, 2, precisions=prec, transpose=(True, True)))
    assert mfa.GEMMKernel.cacheSize() == before + 1
    others = [mfa.GEMMKernel.cached(make(precisions=(P.FP16, P.FP16, P.FP32), transpose=(True, True))),
              mfa.GEMMKernel.cached(make(precisions=(P.BF16, P.BF16, P.BF16), transpose=(True, True))),
              mfa.GEMMKernel.cached(make(precisions=prec, transpose=(True, False))),
              mfa.GEMMKernel.cached(make(precisions=prec, transpose=(False, True)))]
    handles = {a._handle.value} | {k._handle.value for k in others}
    assert len(handles) == 5 and mfa.GEMMKernel.cacheSize() == before + 5
    del a, b, others                                  # library-owned handles: dropping the wrappers must not free them
    again = mfa.GEMMKernel.cached(make(precisions=prec, transpose=(True, True)))
    assert again.threadgroupSize == 192 and mfa.GEMMKernel.cacheSize() == before + 5


def test_encode_without_gpu_fails_loudly_instead_of_falling_back():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    d = make(precisions=(P.BF16, P.BF16, P.FP32))
    for k in (mfa.GEMMKernel.cached(d), mfa.GEMMKernel(mfa.GEMMKernelDescriptor(make()))):
        with pytest.raises(mfa.MFAError) as err:
            k.encode(constants(d), [16, 16, 16])
        assert err.value.status == -6 and "no CPU fallback" in str(err.value)    # MFA_ERROR_NO_DEVICE


def test_cpp_host_mirror_runs_a_gemm_descriptor(tmp_path):
    """metal-flash-attention_b200/host/FlashAttention.hpp: the GEMM types build with g++ against the C ABI and reproduce
    the descriptor -> kernel flow, including the reference's message for an incomplete descriptor."""
    src = tmp_path / "gemm.cpp"
    src.write_text(r'''
#include <cstdio>
#include "metal-flash-attention_b200/host/FlashAttention.hpp"
using namespace FlashAttention;
int main() {
  GEMMDescriptor d;
  d.matrixDimensions = GEMMMatrixDimensions{1000, 600, 300};
  d.memoryPrecisions = GEMMPrecisions{GEMMOperandPrecision::BF16, GEMMOperandPrecision::BF16, GEMMOperandPrecision::FP32};
  d.transposeState = GEMMTransposeState{false, true};
  GEMMKernel k(GEMMKernelDescriptor{d});
  auto [bm, bn, bk] = k.blockDimensions();
  mfa_gemm_function_constants_t c;
  d.setFunctionConstants(c);
  GEMMKernel::register_(d);
  GEMMKernel cached = GEMMKernel::cached(d);
  std::printf("%u %u %u %u %u %u %s\n", bm, bn, bk, k.threadgroupSize(), k.gridSize(c), cached.launchCount(c),
              cached.sourceName().c_str());
  try {
    GEMMKernelDescriptor incomplete{GEMMDescriptor{}};
  } catch (const std::runtime_error &e) {
    std::printf("%s\n", e.what());
  }
  return 0;
}
''')
    exe = tmp_path / "gemm"
    libdir = os.path.dirname(mfa.library_path())
    subprocess.check_call(["g++", "-std=c++17", "-I", ROOT, str(src), "-o", str(exe), "-L", libdir, "-lmfa_b200",
                           f"-Wl,-rpath,{libdir}"])
    out = subprocess.check_output([str(exe)], text=True).splitlines()
    assert out == ["128 256 64 192 24 3 gemm_tcgen05<bfloat, bfloat, float, NT>", "Descriptor was incomplete."]
