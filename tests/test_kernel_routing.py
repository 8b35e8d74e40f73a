"""Which kernel serves a descriptor, and what the kernel object reports about it, pinned over a grid of descriptors.

For every (kernel type, precision policy, transpose state, head dimension, R x C) the grid records the kernel object's
backend, source name, block dimensions, threadgroup size and shared memory -- or the MFAError a rejected descriptor
raises -- and, for batch counts 1, 3 and 64, gridSize and launchCount, with the parameter table's split policy and with
splitPolicy = (0, 1) (never split).  launchCount depends on the SM count, which is 148 both on a B200 and without a
device (the library's fallback), so the fixture holds on either machine.

The fixture is tests/golden/kernel_routing.json; `python -m tests.test_kernel_routing --write` regenerates it."""
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kernel_routing.json")

HEADS = (3, 8, 40, 64, 72, 96, 128, 136, 192, 256, 264)
POLICIES = ("fp32", "fp16", "bf16", "fp16+bf16dO")  # all-FP32, all-FP16, all-BF16, the reference's FP16 Q/K/V + BF16 dO
TRANSPOSES = ((False,) * 4, (True, False, False, False), (False, True, False, False), (False, False, True, False),
              (False, False, False, True), (True,) * 4)
SHAPES = ((64, 64), (77, 64), (64, 77), (256, 2048), (1, 4096), (4096, 4096))
BATCHES = (1, 3, 64)


def _descriptor(policy, R, C, D, transpose):
    import mfa_b200 as mfa
    desc = mfa.AttentionDescriptor()
    desc.lowPrecisionInputs = policy != "fp32"
    if policy == "fp16":
        desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.FP16
    elif policy == "bf16":
        desc.inputPrecisionOverride = mfa.GEMMOperandPrecision.BF16
    desc.matrixDimensions = (R, C, D)
    desc.transposeState = transpose
    return desc


def _kernel(desc, type, split_policy):
    """(properties or ["MFAError", status, message], kernel or None)"""
    import mfa_b200 as mfa
    try:
        kd = desc.kernelDescriptor(type)
        if split_policy is not None:
            kd.splitPolicy = split_policy
        kernel = mfa.AttentionKernel(kd)
    except mfa.MFAError as e:
        return ["MFAError", e.status, e.message], None
    props = [int(kd.backend), kernel.sourceName(), list(kernel.blockDimensions),
             kernel.threadgroupSize, kernel.threadgroupMemoryAllocation]
    return props, kernel


def _per_batch(desc, kernel, method):
    import mfa_b200 as mfa
    out = []
    for batch in BATCHES:
        desc.batchCount = batch
        constants = mfa.FunctionConstantValues()
        desc.setFunctionConstants(constants)
        out.append(getattr(kernel, method)(constants))
    desc.batchCount = 1
    return out


def routing_table():
    """{"kernels": [distinct properties / errors], "cases": {"type|policy|transpose|D": [one entry per shape]}}; an entry
    is [kernel index (table policy), kernel index (split (0, 1)), gridSize x3, launchCount x3 (table), launchCount x3
    (split (0, 1))], or [error index] when the descriptor is rejected."""
    import mfa_b200 as mfa
    kernels, index = [], {}

    def intern(props):
        key = json.dumps(props)
        if key not in index:
            index[key] = len(kernels)
            kernels.append(props)
        return index[key]

    cases = {}
    for type in mfa.AttentionKernelType:
        for policy in POLICIES:
            for transpose in TRANSPOSES:
                for D in HEADS:
                    row = []
                    for R, C in SHAPES:
                        desc = _descriptor(policy, R, C, D, transpose)
                        props, kernel = _kernel(desc, type, None)
                        if kernel is None:
                            row.append([intern(props)])
                            continue
                        props01, kernel01 = _kernel(desc, type, (0, 1))
                        entry = [intern(props), intern(props01)] + _per_batch(desc, kernel, "gridSize")
                        entry += _per_batch(desc, kernel, "launchCount")
                        entry += _per_batch(desc, kernel01, "launchCount") if kernel01 is not None else [None] * 3
                        row.append(entry)
                    key = "|".join([type.name, policy, "".join("T" if t else "-" for t in transpose), str(D)])
                    cases[key] = row
    return {"kernels": kernels, "cases": cases}


def _decode(table, key, i):
    entry = table["cases"][key][i]
    resolved = [table["kernels"][entry[0]]]
    if len(entry) > 1:
        resolved.append(table["kernels"][entry[1]])
        resolved += entry[2:]
    return resolved


def test_kernel_routing_matches_fixture():
    with open(GOLDEN) as f:
        expected = json.load(f)
    actual = routing_table()
    assert sorted(actual["cases"]) == sorted(expected["cases"])
    mismatches = []
    for key in expected["cases"]:
        for i, (R, C) in enumerate(SHAPES):
            want, got = _decode(expected, key, i), _decode(actual, key, i)
            if want != got:
                mismatches.append(f"{key} R={R} C={C}: expected {want}, got {got}")
    assert not mismatches, f"{len(mismatches)} routing differences, first: " + "\n".join(mismatches[:10])


if __name__ == "__main__":
    import sys
    if sys.argv[1:] != ["--write"]:
        sys.exit("usage: python -m tests.test_kernel_routing --write")
    with open(GOLDEN, "w") as f:
        table = routing_table()
        f.write('{"kernels": [\n' + ",\n".join(json.dumps(k) for k in table["kernels"]) + '],\n"cases": {\n')
        f.write(",\n".join(f"{json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}" for k, v in table["cases"].items()))
        f.write("}}\n")
