"""mfa_b200 -- Python mirror of the reference's Swift attention API over the C ABI.

The reference (philipturner/metal-flash-attention) is a Swift package; Swift is not installed in this
image, so the host-side mirror used by tests/ and bench.py is this thin ctypes layer.  It keeps the
reference's names, field meanings and failure behaviour:

    AttentionDescriptor            Sources/FlashAttention/Attention/AttentionDescriptor/AttentionDescriptor.swift:10-27
      .kernelDescriptor(type:)     :33-130
      .setFunctionConstants(_:)    :139-148
      .memoryPrecisions            AttentionDescriptor+Precisions.swift:10-146
      .registerPrecisions          :149-215
    AttentionKernelDescriptor      Attention/AttentionKernelDescriptor.swift:7-48
    AttentionKernelType            Attention/AttentionKernelType.swift:8-23
    AttentionOperand(.bufferBinding)  Attention/AttentionOperand.swift:8-72
    AttentionKernel                Attention/AttentionKernel/AttentionKernel.swift:11-50, 268-363
    GEMMOperandPrecision           GEMM/GEMMOperandPrecision.swift:33-61
    GEMMDescriptor                 GEMM/GEMMDescriptor/GEMMDescriptor.swift:10-44
      .setFunctionConstants(_:)    :327-380
    GEMMKernelDescriptor           GEMM/GEMMKernelDescriptor.swift:21-181; (descriptor:) GEMMDescriptor.swift:106-234
    GEMMKernel                     GEMM/GEMMKernel/GEMMKernel.swift:10-270
      .register / pipelineCache    GEMM/GEMMDescriptor/GEMMDescriptor+PipelineCache.swift:16-36

All arithmetic happens in libmfa_b200.so (hand-written sm_100a CUDA).  There is no Python or CPU
fallback: if the shared library is missing, importing this package raises.  Where the reference traps
with fatalError(...), this mirror raises MFAError carrying the same message.
"""
from __future__ import annotations

import ctypes
import enum
import os
from typing import Dict, Optional, Sequence, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("MFA_B200_LIBRARY") or os.path.join(_HERE, "lib", "libmfa_b200.so")  # override: tuning builds only

MFA_OPERAND_COUNT = 14
MFA_BUFFER_COUNT = 10
MFA_GEMM_BUFFER_COUNT = 3


class MFAError(RuntimeError):
    """Raised where the reference would fatalError(); .status is the mfa_status_t code."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[mfa status {status}] {message}")
        self.status = status
        self.message = message


# -------------------------------------------------------------------------------------------------
# C structs (must match include/mfa_b200.h)
# -------------------------------------------------------------------------------------------------
class _CDescriptor(ctypes.Structure):
    _fields_ = [
        ("low_precision_inputs", ctypes.c_uint8),
        ("low_precision_intermediates", ctypes.c_uint8),
        ("has_matrix_dimensions", ctypes.c_uint8),
        ("has_transpose_state", ctypes.c_uint8),
        ("row", ctypes.c_uint32),
        ("column", ctypes.c_uint32),
        ("head", ctypes.c_uint16),
        ("transpose_Q", ctypes.c_uint8),
        ("transpose_K", ctypes.c_uint8),
        ("transpose_V", ctypes.c_uint8),
        ("transpose_O", ctypes.c_uint8),
        ("input_precision_override", ctypes.c_uint8),
        ("reserved0", ctypes.c_uint8),
        ("batch_count", ctypes.c_uint32),
    ]


class _CKernelDescriptor(ctypes.Structure):
    _fields_ = [
        ("has_block_dimensions", ctypes.c_uint8),
        ("block_parallelization", ctypes.c_uint16),
        ("block_traversal", ctypes.c_uint16),
        ("block_head", ctypes.c_uint16),
        ("cache_state_valid_mask", ctypes.c_uint16),
        ("cache_state_mask", ctypes.c_uint16),
        ("has_head_dimension", ctypes.c_uint8),
        ("head_dimension", ctypes.c_uint16),
        ("memory_precisions", ctypes.c_uint8 * MFA_OPERAND_COUNT),
        ("register_precisions", ctypes.c_uint8 * MFA_OPERAND_COUNT),
        ("prefer_async_cache", ctypes.c_uint8),
        ("prefer_async_load", ctypes.c_uint8),
        ("transpose_state_valid_mask", ctypes.c_uint16),
        ("transpose_state_mask", ctypes.c_uint16),
        ("type", ctypes.c_uint8),
        ("backend", ctypes.c_uint8),
        ("exp2_fma_quarters", ctypes.c_uint8),
        ("split_min_blocks", ctypes.c_uint8),
        ("split_max", ctypes.c_uint8),
    ]


class _CFunctionConstants(ctypes.Structure):
    _fields_ = [("row", ctypes.c_uint32), ("column", ctypes.c_uint32), ("batch_count", ctypes.c_uint32)]


class _CGEMMDescriptor(ctypes.Structure):
    _fields_ = [
        ("batch_dimension", ctypes.c_uint32),
        ("has_leading_dimensions", ctypes.c_uint8),
        ("load_previous_C", ctypes.c_uint8),
        ("has_matrix_dimensions", ctypes.c_uint8),
        ("has_memory_precisions", ctypes.c_uint8),
        ("has_transpose_state", ctypes.c_uint8),
        ("transpose_A", ctypes.c_uint8),
        ("transpose_B", ctypes.c_uint8),
        ("memory_precisions", ctypes.c_uint8 * 3),
        ("leading_dimensions", ctypes.c_uint32 * 3),
        ("M", ctypes.c_uint32),
        ("N", ctypes.c_uint32),
        ("K", ctypes.c_uint32),
    ]


class _CGEMMFunctionConstants(ctypes.Structure):
    _fields_ = [
        ("M", ctypes.c_uint32),
        ("N", ctypes.c_uint32),
        ("K", ctypes.c_uint32),
        ("leading_dimensions", ctypes.c_uint32 * 3),
        ("load_previous_C", ctypes.c_uint8),
        ("batch_count", ctypes.c_uint32),
    ]


class _CGEMMKernelDescriptor(ctypes.Structure):
    _fields_ = [
        ("has_block_dimensions", ctypes.c_uint8),
        ("block_dimensions", ctypes.c_uint16 * 3),
        ("has_leading_block_dimensions", ctypes.c_uint8),
        ("leading_block_dimensions", ctypes.c_uint16 * 3),
        ("has_memory_precisions", ctypes.c_uint8),
        ("memory_precisions", ctypes.c_uint8 * 3),
        ("has_register_precisions", ctypes.c_uint8),
        ("register_precisions", ctypes.c_uint8 * 3),
        ("prefer_async_load", ctypes.c_uint8),
        ("prefer_async_store", ctypes.c_uint8),
        ("has_splits", ctypes.c_uint8),
        ("splits", ctypes.c_uint16 * 2),
        ("has_transpose_state", ctypes.c_uint8),
        ("transpose_A", ctypes.c_uint8),
        ("transpose_B", ctypes.c_uint8),
        ("backend", ctypes.c_uint8),
    ]


def _load():
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is deliberately no Python/CPU fallback for the attention kernels)")
    lib = ctypes.CDLL(_LIB_PATH)
    c = ctypes
    lib.mfa_last_error.restype = c.c_char_p
    lib.mfa_version.restype = c.c_char_p
    lib.mfa_precision_name.restype = c.c_char_p
    lib.mfa_operand_name.restype = c.c_char_p
    lib.mfa_attention_kernel_source_name.restype = c.c_char_p
    lib.mfa_attention_kernel_source_name.argtypes = [c.c_void_p]
    lib.mfa_attention_descriptor_parameter_file.restype = c.c_char_p
    lib.mfa_attention_descriptor_parameter_file.argtypes = [c.POINTER(_CDescriptor), c.c_int]
    lib.mfa_attention_descriptor_memory_precision.argtypes = [c.POINTER(_CDescriptor), c.c_int, c.POINTER(c.c_int)]
    lib.mfa_attention_descriptor_register_precision.argtypes = [c.POINTER(_CDescriptor), c.c_int, c.POINTER(c.c_int)]
    lib.mfa_attention_descriptor_kernel_descriptor.argtypes = [c.POINTER(_CDescriptor), c.c_int,
                                                               c.POINTER(_CKernelDescriptor)]
    lib.mfa_attention_descriptor_set_function_constants.argtypes = [c.POINTER(_CDescriptor),
                                                                    c.POINTER(_CFunctionConstants)]
    lib.mfa_attention_descriptor_operand_elements.argtypes = [c.POINTER(_CDescriptor), c.c_int,
                                                              c.POINTER(c.c_size_t)]
    lib.mfa_attention_kernel_descriptor_init.argtypes = [c.POINTER(_CKernelDescriptor)]
    lib.mfa_attention_kernel_create.argtypes = [c.POINTER(_CKernelDescriptor), c.POINTER(c.c_void_p)]
    lib.mfa_attention_kernel_destroy.argtypes = [c.c_void_p]
    lib.mfa_attention_kernel_destroy.restype = None
    lib.mfa_attention_kernel_block_dimensions.argtypes = [c.c_void_p, c.POINTER(c.c_uint16 * 3)]
    lib.mfa_attention_kernel_threadgroup_size.argtypes = [c.c_void_p, c.POINTER(c.c_uint32)]
    lib.mfa_attention_kernel_threadgroup_memory_allocation.argtypes = [c.c_void_p, c.POINTER(c.c_uint32)]
    lib.mfa_attention_kernel_grid_size.argtypes = [c.c_void_p, c.POINTER(_CFunctionConstants), c.POINTER(c.c_uint32)]
    lib.mfa_attention_kernel_launch_count.argtypes = [c.c_void_p, c.POINTER(_CFunctionConstants),
                                                      c.POINTER(c.c_uint32)]
    lib.mfa_attention_kernel_encode.argtypes = [c.c_void_p, c.POINTER(_CFunctionConstants),
                                                c.POINTER(c.c_void_p * MFA_BUFFER_COUNT), c.c_void_p]
    lib.mfa_attention_kernel_cache_fetch.argtypes = [c.POINTER(_CDescriptor), c.c_int, c.POINTER(c.c_void_p)]
    lib.mfa_attention_kernel_cache_size.restype = c.c_int
    lib.mfa_attention_run_host.argtypes = [c.POINTER(_CDescriptor), c.c_uint32,
                                           c.POINTER(c.c_void_p * MFA_BUFFER_COUNT), c.c_int]
    lib.mfa_gemm_descriptor_init.argtypes = [c.POINTER(_CGEMMDescriptor)]
    lib.mfa_gemm_descriptor_init.restype = None
    lib.mfa_gemm_descriptor_set_function_constants.argtypes = [c.POINTER(_CGEMMDescriptor),
                                                               c.POINTER(_CGEMMFunctionConstants)]
    lib.mfa_gemm_kernel_descriptor_init.argtypes = [c.POINTER(_CGEMMKernelDescriptor)]
    lib.mfa_gemm_kernel_descriptor_init.restype = None
    lib.mfa_gemm_descriptor_kernel_descriptor.argtypes = [c.POINTER(_CGEMMDescriptor), c.POINTER(_CGEMMKernelDescriptor)]
    lib.mfa_gemm_kernel_create.argtypes = [c.POINTER(_CGEMMKernelDescriptor), c.POINTER(c.c_void_p)]
    lib.mfa_gemm_kernel_destroy.argtypes = [c.c_void_p]
    lib.mfa_gemm_kernel_destroy.restype = None
    lib.mfa_gemm_kernel_block_dimensions.argtypes = [c.c_void_p, c.POINTER(c.c_uint16 * 3)]
    lib.mfa_gemm_kernel_threadgroup_size.argtypes = [c.c_void_p, c.POINTER(c.c_uint32)]
    lib.mfa_gemm_kernel_threadgroup_memory_allocation.argtypes = [c.c_void_p, c.POINTER(c.c_uint32)]
    lib.mfa_gemm_kernel_grid_size.argtypes = [c.c_void_p, c.POINTER(_CGEMMFunctionConstants), c.POINTER(c.c_uint32)]
    lib.mfa_gemm_kernel_launch_count.argtypes = [c.c_void_p, c.POINTER(_CGEMMFunctionConstants), c.POINTER(c.c_uint32)]
    lib.mfa_gemm_kernel_source_name.argtypes = [c.c_void_p]
    lib.mfa_gemm_kernel_source_name.restype = c.c_char_p
    lib.mfa_gemm_kernel_encode.argtypes = [c.c_void_p, c.POINTER(_CGEMMFunctionConstants),
                                           c.POINTER(c.c_void_p * MFA_GEMM_BUFFER_COUNT), c.c_void_p]
    lib.mfa_gemm_kernel_cache_fetch.argtypes = [c.POINTER(_CGEMMDescriptor), c.POINTER(c.c_void_p)]
    lib.mfa_gemm_kernel_cache_size.restype = c.c_int
    try:
        lib.mfa_set_parameter_table.argtypes = [c.c_int, c.c_int, c.c_char_p]
        lib.mfa_host_alloc.argtypes = [c.c_size_t, c.c_int, c.POINTER(c.c_void_p)]
        lib.mfa_host_alloc_upload.argtypes = [c.c_size_t, c.c_int, c.POINTER(c.c_void_p)]
        lib.mfa_host_free.argtypes = [c.c_void_p]
        lib.mfa_host_bind_thread_to_device.argtypes = [c.c_int, c.POINTER(c.c_int)]
        lib.mfa_release_device_resources.argtypes = [c.c_int]
    except AttributeError:
        # only an older tuning build selected through MFA_B200_LIBRARY can lack these (A/B timing against it still works)
        if not os.environ.get("MFA_B200_LIBRARY"):
            raise
    return lib


_lib = _load()


def _check(status: int):
    if status != 0:
        raise MFAError(status, _lib.mfa_last_error().decode())


def hostAlloc(nbytes: int, device: int = 0, upload: bool = False) -> int:
    """mfa_host_alloc: page-locked host buffer on the NUMA node of `device` (for runHost); returns the address.
    upload=True (mfa_host_alloc_upload): write-combined pages for buffers the host only writes (Q, K, V, dO)."""
    out = ctypes.c_void_p()
    _check((_lib.mfa_host_alloc_upload if upload else _lib.mfa_host_alloc)(int(nbytes), int(device), ctypes.byref(out)))
    return out.value


def hostFree(address: int) -> None:
    _check(_lib.mfa_host_free(ctypes.c_void_p(address)))


def bindThreadToDevice(device: int = 0) -> int:
    """mfa_host_bind_thread_to_device: pin the calling thread to the CPUs of the GPU's NUMA node; returns the node
    (-1: the platform reports none, nothing changed)."""
    node = ctypes.c_int(-1)
    _check(_lib.mfa_host_bind_thread_to_device(int(device), ctypes.byref(node)))
    return node.value


def releaseDeviceResources(device: int = 0) -> None:
    """mfa_release_device_resources: free the library's scratch and workspaces on `device`."""
    _check(_lib.mfa_release_device_resources(int(device)))


def setParameterTable(type: "AttentionKernelType", text: Optional[str], transposed: bool = False) -> None:
    """mfa_set_parameter_table: replace (text) or restore (None) the tcgen05-family parameter table of `type`."""
    _check(_lib.mfa_set_parameter_table(int(type), int(bool(transposed)),
                                        None if text is None else text.encode()))


def maxExp2FmaQuarters(type: "AttentionKernelType") -> int:
    return _lib.mfa_max_exp2_fma_quarters(int(type))


def library_path() -> str:
    return _LIB_PATH


def version() -> str:
    return _lib.mfa_version().decode()


# -------------------------------------------------------------------------------------------------
# Enumerations
# -------------------------------------------------------------------------------------------------
class GEMMOperandPrecision(enum.IntEnum):
    """GEMMOperandPrecision.swift:33-61 (raw values are ABI)."""
    FP32 = 0
    FP16 = 1
    BF16 = 2

    @property
    def size(self) -> int:
        return 4 if self == GEMMOperandPrecision.FP32 else 2


class AttentionKernelType(enum.IntEnum):
    """AttentionKernelType.swift:8-23."""
    forward = 0
    backwardQuery = 1
    backwardKeyValue = 2


class AttentionOperand(enum.IntEnum):
    """AttentionOperand.swift:8-72; values 0..9 are the buffer bindings."""
    Q = 0
    K = 1
    V = 2
    O = 3
    L = 4
    D = 5
    dO = 6
    dV = 7
    dK = 8
    dQ = 9
    S = 10
    P = 11
    dP = 12
    dS = 13

    @property
    def bufferBinding(self) -> Optional[int]:
        return int(self) if int(self) < MFA_BUFFER_COUNT else None

    @property
    def description(self) -> str:
        return self.name


class Backend(enum.IntEnum):
    simtFP32 = 0
    tcgen05 = 1


# -------------------------------------------------------------------------------------------------
# AttentionDescriptor
# -------------------------------------------------------------------------------------------------
class AttentionDescriptor:
    """AttentionDescriptor.swift:10-27.  `matrixDimensions = (row, column, head)`,
    `transposeState = (Q, K, V, O)`; both start as None (Swift optionals)."""

    def __init__(self):
        self.lowPrecisionInputs: bool = False
        self.lowPrecisionIntermediates: bool = False
        self.matrixDimensions: Optional[Tuple[int, int, int]] = None
        self.transposeState: Optional[Tuple[bool, bool, bool, bool]] = None
        # B200 extensions (include/mfa_b200.h): None = reference policy (FP16 inputs).
        self.inputPrecisionOverride: Optional[GEMMOperandPrecision] = None
        self.batchCount: int = 1

    def _c(self) -> _CDescriptor:
        d = _CDescriptor()
        d.low_precision_inputs = int(bool(self.lowPrecisionInputs))
        d.low_precision_intermediates = int(bool(self.lowPrecisionIntermediates))
        if self.matrixDimensions is not None:
            d.has_matrix_dimensions = 1
            d.row, d.column, d.head = (int(x) for x in self.matrixDimensions)
        if self.transposeState is not None:
            d.has_transpose_state = 1
            d.transpose_Q, d.transpose_K, d.transpose_V, d.transpose_O = (int(bool(x)) for x in self.transposeState)
        d.input_precision_override = int(self.inputPrecisionOverride) if self.inputPrecisionOverride else 0
        d.batch_count = int(self.batchCount)
        return d

    @property
    def memoryPrecisions(self) -> Dict[AttentionOperand, GEMMOperandPrecision]:
        c, out = self._c(), {}
        for op in list(AttentionOperand)[:MFA_BUFFER_COUNT]:
            value = ctypes.c_int()
            _check(_lib.mfa_attention_descriptor_memory_precision(ctypes.byref(c), int(op), ctypes.byref(value)))
            out[op] = GEMMOperandPrecision(value.value)
        return out

    @property
    def registerPrecisions(self) -> Dict[AttentionOperand, GEMMOperandPrecision]:
        c, out = self._c(), {}
        for op in AttentionOperand:
            value = ctypes.c_int()
            _check(_lib.mfa_attention_descriptor_register_precision(ctypes.byref(c), int(op), ctypes.byref(value)))
            out[op] = GEMMOperandPrecision(value.value)
        return out

    def parameterFile(self, type: AttentionKernelType) -> str:
        c = self._c()
        return _lib.mfa_attention_descriptor_parameter_file(ctypes.byref(c), int(type)).decode()

    def kernelDescriptor(self, type: AttentionKernelType) -> "AttentionKernelDescriptor":
        c = self._c()
        out = AttentionKernelDescriptor()
        _check(_lib.mfa_attention_descriptor_kernel_descriptor(ctypes.byref(c), int(type), ctypes.byref(out._c)))
        return out

    def setFunctionConstants(self, constants: "FunctionConstantValues") -> None:
        c = self._c()
        _check(_lib.mfa_attention_descriptor_set_function_constants(ctypes.byref(c), ctypes.byref(constants._c)))

    def operandElements(self, operand: AttentionOperand) -> int:
        c, n = self._c(), ctypes.c_size_t()
        _check(_lib.mfa_attention_descriptor_operand_elements(ctypes.byref(c), int(operand), ctypes.byref(n)))
        return n.value

    def runHost(self, types: Sequence[AttentionKernelType], hostBuffers: Dict[AttentionOperand, int],
                device: int = 0) -> None:
        """End-to-end call on HOST pointers (mfa_attention_run_host): H2D -> kernels -> D2H."""
        c = self._c()
        mask = 0
        for t in types:
            mask |= 1 << int(t)
        arr = (ctypes.c_void_p * MFA_BUFFER_COUNT)()
        for op, ptr in hostBuffers.items():
            arr[int(op)] = ptr
        _check(_lib.mfa_attention_run_host(ctypes.byref(c), mask, ctypes.byref(arr), device))


class FunctionConstantValues:
    """Stand-in for MTLFunctionConstantValues: R at index 0, C at index 1 (AttentionDescriptor.swift:144-147)."""

    def __init__(self):
        self._c = _CFunctionConstants()

    @property
    def row(self) -> int:
        return self._c.row

    @property
    def column(self) -> int:
        return self._c.column

    @property
    def batchCount(self) -> int:
        return self._c.batch_count


# -------------------------------------------------------------------------------------------------
# AttentionKernelDescriptor
# -------------------------------------------------------------------------------------------------
class AttentionKernelDescriptor:
    """AttentionKernelDescriptor.swift:7-48 (a plain, editable value)."""

    def __init__(self):
        self._c = _CKernelDescriptor()
        _lib.mfa_attention_kernel_descriptor_init(ctypes.byref(self._c))

    @property
    def blockDimensions(self) -> Optional[Tuple[int, int, int]]:
        if not self._c.has_block_dimensions:
            return None
        return (self._c.block_parallelization, self._c.block_traversal, self._c.block_head)

    @blockDimensions.setter
    def blockDimensions(self, value):
        if value is None:
            self._c.has_block_dimensions = 0
        else:
            self._c.has_block_dimensions = 1
            self._c.block_parallelization, self._c.block_traversal, self._c.block_head = (int(v) for v in value)

    @property
    def cacheState(self) -> Dict[AttentionOperand, bool]:
        return {op: bool((self._c.cache_state_mask >> int(op)) & 1) for op in AttentionOperand
                if (self._c.cache_state_valid_mask >> int(op)) & 1}

    @property
    def headDimension(self) -> Optional[int]:
        return self._c.head_dimension if self._c.has_head_dimension else None

    @headDimension.setter
    def headDimension(self, value):
        self._c.has_head_dimension = 0 if value is None else 1
        self._c.head_dimension = 0 if value is None else int(value)

    def _precisions(self, array) -> Dict[AttentionOperand, GEMMOperandPrecision]:
        return {op: GEMMOperandPrecision(array[int(op)]) for op in AttentionOperand if array[int(op)] != 0xFF}

    @property
    def memoryPrecisions(self):
        return self._precisions(self._c.memory_precisions)

    @property
    def registerPrecisions(self):
        return self._precisions(self._c.register_precisions)

    def setMemoryPrecision(self, operand: AttentionOperand, precision: Optional[GEMMOperandPrecision]):
        self._c.memory_precisions[int(operand)] = 0xFF if precision is None else int(precision)

    def setRegisterPrecision(self, operand: AttentionOperand, precision: Optional[GEMMOperandPrecision]):
        self._c.register_precisions[int(operand)] = 0xFF if precision is None else int(precision)

    @property
    def preferAsyncCache(self) -> Optional[bool]:
        return None if self._c.prefer_async_cache == 0xFF else bool(self._c.prefer_async_cache)

    @preferAsyncCache.setter
    def preferAsyncCache(self, value):
        self._c.prefer_async_cache = 0xFF if value is None else int(bool(value))

    @property
    def preferAsyncLoad(self) -> Optional[bool]:
        return None if self._c.prefer_async_load == 0xFF else bool(self._c.prefer_async_load)

    @preferAsyncLoad.setter
    def preferAsyncLoad(self, value):
        self._c.prefer_async_load = 0xFF if value is None else int(bool(value))

    @property
    def transposeState(self) -> Dict[AttentionOperand, bool]:
        return {op: bool((self._c.transpose_state_mask >> int(op)) & 1) for op in AttentionOperand
                if (self._c.transpose_state_valid_mask >> int(op)) & 1}

    @property
    def type(self) -> Optional[AttentionKernelType]:
        return None if self._c.type == 0xFF else AttentionKernelType(self._c.type)

    @type.setter
    def type(self, value):
        self._c.type = 0xFF if value is None else int(value)

    @property
    def backend(self) -> Backend:
        return Backend(self._c.backend)

    @backend.setter
    def backend(self, value):
        self._c.backend = int(value)

    # ---- B200 extension: the tuning columns of the parameter-table row (plain, editable data like blockDimensions)
    @property
    def exp2FmaQuarters(self) -> int:
        """Of every 4 element pairs of P, how many take exp2 on the FMA pipe: selects the kernel instantiation."""
        return self._c.exp2_fma_quarters

    @exp2FmaQuarters.setter
    def exp2FmaQuarters(self, value):
        self._c.exp2_fma_quarters = int(value)

    @property
    def splitPolicy(self) -> Tuple[int, int]:
        """(minimum blocks per traversal range, maximum ranges) for small grids; minimum 0 = never split."""
        return (self._c.split_min_blocks, self._c.split_max)

    @splitPolicy.setter
    def splitPolicy(self, value):
        self._c.split_min_blocks, self._c.split_max = (int(v) for v in value)


# -------------------------------------------------------------------------------------------------
# AttentionKernel
# -------------------------------------------------------------------------------------------------
class AttentionKernel:
    """AttentionKernel.swift:11-50.  `encode` performs what the reference's callers do by hand
    (makeLibrary / makeComputePipelineState / setBuffer x10 / dispatchThreadgroups,
    SquareAttentionTest.swift:240-372) against DEVICE pointers."""

    def __init__(self, descriptor: AttentionKernelDescriptor):
        self._handle = ctypes.c_void_p()
        self._owned = True
        _check(_lib.mfa_attention_kernel_create(ctypes.byref(descriptor._c), ctypes.byref(self._handle)))

    @classmethod
    def cached(cls, descriptor: AttentionDescriptor, type: AttentionKernelType) -> "AttentionKernel":
        """mfa_attention_kernel_cache_fetch: the kernel object for (descriptor, type), built once per process and
        owned by the library (the analogue of GEMMKernel.pipelineCache, GEMMDescriptor+PipelineCache.swift:16-36)."""
        self = cls.__new__(cls)
        self._handle = ctypes.c_void_p()
        self._owned = False
        c = descriptor._c()
        _check(_lib.mfa_attention_kernel_cache_fetch(ctypes.byref(c), int(type), ctypes.byref(self._handle)))
        return self

    @staticmethod
    def cacheSize() -> int:
        return _lib.mfa_attention_kernel_cache_size()

    def __del__(self):
        handle = getattr(self, "_handle", None)
        if handle and getattr(self, "_owned", False) and _lib is not None:  # _lib is None during interpreter teardown
            _lib.mfa_attention_kernel_destroy(handle)
            self._handle = None

    @property
    def blockDimensions(self) -> Tuple[int, int, int]:
        out = (ctypes.c_uint16 * 3)()
        _check(_lib.mfa_attention_kernel_block_dimensions(self._handle, ctypes.byref(out)))
        return (out[0], out[1], out[2])

    @property
    def threadgroupSize(self) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_attention_kernel_threadgroup_size(self._handle, ctypes.byref(out)))
        return out.value

    @property
    def threadgroupMemoryAllocation(self) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_attention_kernel_threadgroup_memory_allocation(self._handle, ctypes.byref(out)))
        return out.value

    def gridSize(self, constants: FunctionConstantValues) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_attention_kernel_grid_size(self._handle, ctypes.byref(constants._c), ctypes.byref(out)))
        return out.value

    def launchCount(self, constants: FunctionConstantValues) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_attention_kernel_launch_count(self._handle, ctypes.byref(constants._c), ctypes.byref(out)))
        return out.value

    def sourceName(self) -> str:
        """Stands in for createSource() (AttentionKernel+Source.swift:11-55): the kernels are AOT-compiled."""
        return _lib.mfa_attention_kernel_source_name(self._handle).decode()

    def encode(self, constants: FunctionConstantValues, buffers: Dict[AttentionOperand, int],
               stream: int = 0) -> None:
        """buffers: {AttentionOperand: device pointer}; stream: cudaStream_t as int (0 = default)."""
        arr = (ctypes.c_void_p * MFA_BUFFER_COUNT)()
        for op, ptr in buffers.items():
            binding = AttentionOperand(op).bufferBinding
            if binding is None:
                raise MFAError(-2, f"Operand {AttentionOperand(op).name} has no buffer binding.")
            arr[binding] = ptr
        _check(_lib.mfa_attention_kernel_encode(self._handle, ctypes.byref(constants._c), ctypes.byref(arr),
                                                ctypes.c_void_p(stream)))


# -------------------------------------------------------------------------------------------------
# GEMM: GEMMDescriptor, GEMMKernelDescriptor, GEMMKernel
# -------------------------------------------------------------------------------------------------
def _triple(values, cast=int):
    return tuple(cast(v) for v in values)


class GEMMDescriptor:
    """GEMMDescriptor.swift:10-44.  C = A . B (or C += A . B with loadPreviousC).  `matrixDimensions = (M, N, K)`,
    `memoryPrecisions = (A, B, C)`, `transposeState = (A, B)`, `leadingDimensions = (A, B, C)`; the optionals start as
    None.  batchDimension > 1 (B200 extension): independent problems stored back to back."""

    def __init__(self):
        self.batchDimension: int = 1
        self.leadingDimensions: Optional[Tuple[int, int, int]] = None
        self.loadPreviousC: bool = False
        self.matrixDimensions: Optional[Tuple[int, int, int]] = None
        self.memoryPrecisions: Optional[Tuple[GEMMOperandPrecision, GEMMOperandPrecision, GEMMOperandPrecision]] = None
        self.transposeState: Optional[Tuple[bool, bool]] = None

    def _c(self) -> _CGEMMDescriptor:
        d = _CGEMMDescriptor()
        _lib.mfa_gemm_descriptor_init(ctypes.byref(d))
        d.batch_dimension = int(self.batchDimension)
        if self.leadingDimensions is not None:
            d.has_leading_dimensions = 1
            d.leading_dimensions[:] = _triple(self.leadingDimensions)
        d.load_previous_C = int(bool(self.loadPreviousC))
        if self.matrixDimensions is not None:
            d.has_matrix_dimensions = 1
            d.M, d.N, d.K = _triple(self.matrixDimensions)
        if self.memoryPrecisions is not None:
            d.has_memory_precisions = 1
            d.memory_precisions[:] = _triple(self.memoryPrecisions)
        if self.transposeState is not None:
            d.has_transpose_state = 1
            d.transpose_A, d.transpose_B = (int(bool(x)) for x in self.transposeState)
        return d

    def setFunctionConstants(self, constants: "GEMMFunctionConstantValues") -> None:
        """M, N, K, the leading dimensions (chooseLeadingDimension's defaults when None), loadPreviousC, the batch."""
        c = self._c()
        _check(_lib.mfa_gemm_descriptor_set_function_constants(ctypes.byref(c), ctypes.byref(constants._c)))


class GEMMFunctionConstantValues:
    """Stand-in for the MTLFunctionConstantValues GEMMDescriptor.setFunctionConstants fills (indices 0-2, 5-7, 10)."""

    def __init__(self):
        self._c = _CGEMMFunctionConstants()

    @property
    def matrixDimensions(self) -> Tuple[int, int, int]:
        return (self._c.M, self._c.N, self._c.K)

    @property
    def leadingDimensions(self) -> Tuple[int, int, int]:
        return tuple(self._c.leading_dimensions)

    @property
    def loadPreviousC(self) -> bool:
        return bool(self._c.load_previous_C)

    @property
    def batchCount(self) -> int:
        return self._c.batch_count


class GEMMKernelDescriptor:
    """GEMMKernelDescriptor.swift:21-181 (a plain, editable value).  GEMMKernelDescriptor(descriptor) runs this
    library's heuristic (GEMMDescriptor.swift:106-234 analogue); GEMMKernelDescriptor() is the empty one."""

    def __init__(self, descriptor: Optional[GEMMDescriptor] = None):
        self._c = _CGEMMKernelDescriptor()
        _lib.mfa_gemm_kernel_descriptor_init(ctypes.byref(self._c))
        if descriptor is not None:
            d = descriptor._c()
            _check(_lib.mfa_gemm_descriptor_kernel_descriptor(ctypes.byref(d), ctypes.byref(self._c)))

    def _get3(self, flag, array, cast=int):
        return tuple(cast(v) for v in array) if getattr(self._c, flag) else None

    def _set3(self, flag, name, value):
        if value is None:
            setattr(self._c, flag, 0)
        else:
            setattr(self._c, flag, 1)
            getattr(self._c, name)[:] = _triple(value)

    @property
    def blockDimensions(self) -> Optional[Tuple[int, int, int]]:
        return self._get3("has_block_dimensions", self._c.block_dimensions)

    @blockDimensions.setter
    def blockDimensions(self, value):
        self._set3("has_block_dimensions", "block_dimensions", value)

    @property
    def leadingBlockDimensions(self) -> Optional[Tuple[int, int, int]]:
        return self._get3("has_leading_block_dimensions", self._c.leading_block_dimensions)

    @leadingBlockDimensions.setter
    def leadingBlockDimensions(self, value):
        self._set3("has_leading_block_dimensions", "leading_block_dimensions", value)

    @property
    def memoryPrecisions(self):
        return self._get3("has_memory_precisions", self._c.memory_precisions, GEMMOperandPrecision)

    @memoryPrecisions.setter
    def memoryPrecisions(self, value):
        self._set3("has_memory_precisions", "memory_precisions", value)

    @property
    def registerPrecisions(self):
        return self._get3("has_register_precisions", self._c.register_precisions, GEMMOperandPrecision)

    @registerPrecisions.setter
    def registerPrecisions(self, value):
        self._set3("has_register_precisions", "register_precisions", value)

    @property
    def preferAsyncLoad(self) -> bool:
        return bool(self._c.prefer_async_load)

    @preferAsyncLoad.setter
    def preferAsyncLoad(self, value):
        self._c.prefer_async_load = int(bool(value))

    @property
    def preferAsyncStore(self) -> Optional[bool]:
        return None if self._c.prefer_async_store == 0xFF else bool(self._c.prefer_async_store)

    @preferAsyncStore.setter
    def preferAsyncStore(self, value):
        self._c.prefer_async_store = 0xFF if value is None else int(bool(value))

    @property
    def splits(self) -> Optional[Tuple[int, int]]:
        return (self._c.splits[0], self._c.splits[1]) if self._c.has_splits else None

    @splits.setter
    def splits(self, value):
        if value is None:
            self._c.has_splits = 0
        else:
            self._c.has_splits = 1
            self._c.splits[0], self._c.splits[1] = (int(v) for v in value)

    @property
    def transposeState(self) -> Optional[Tuple[bool, bool]]:
        return (bool(self._c.transpose_A), bool(self._c.transpose_B)) if self._c.has_transpose_state else None

    @transposeState.setter
    def transposeState(self, value):
        if value is None:
            self._c.has_transpose_state = 0
        else:
            self._c.has_transpose_state = 1
            self._c.transpose_A, self._c.transpose_B = (int(bool(v)) for v in value)

    @property
    def backend(self) -> Backend:
        return Backend(self._c.backend)

    @backend.setter
    def backend(self, value):
        self._c.backend = int(value)


class GEMMKernel:
    """GEMMKernel.swift:10-270.  `encode` binds A, B, C (device pointers, bindings 0, 1, 2) and dispatches, which the
    reference leaves to its caller (AdversarialShapeTest.swift:140-169)."""

    def __init__(self, descriptor: GEMMKernelDescriptor):
        self._handle = ctypes.c_void_p()
        self._owned = True
        _check(_lib.mfa_gemm_kernel_create(ctypes.byref(descriptor._c), ctypes.byref(self._handle)))

    @classmethod
    def register(cls, descriptor: GEMMDescriptor) -> None:
        """GEMMKernel.register(descriptor:): build the descriptor's kernel object once (GEMMDescriptor+PipelineCache.swift:
        24-36)."""
        cls.cached(descriptor)

    @classmethod
    def cached(cls, descriptor: GEMMDescriptor) -> "GEMMKernel":
        """pipelineCache[descriptor]: the library-owned kernel object (mfa_gemm_kernel_cache_fetch).  The key is the
        precisions and transposes; M, N, K, leading dimensions, loadPreviousC and the batch are launch constants."""
        self = cls.__new__(cls)
        self._handle = ctypes.c_void_p()
        self._owned = False
        c = descriptor._c()
        _check(_lib.mfa_gemm_kernel_cache_fetch(ctypes.byref(c), ctypes.byref(self._handle)))
        return self

    @staticmethod
    def cacheSize() -> int:
        return _lib.mfa_gemm_kernel_cache_size()

    def __del__(self):
        handle = getattr(self, "_handle", None)
        if handle and getattr(self, "_owned", False) and _lib is not None:
            _lib.mfa_gemm_kernel_destroy(handle)
            self._handle = None

    @property
    def blockDimensions(self) -> Tuple[int, int, int]:
        out = (ctypes.c_uint16 * 3)()
        _check(_lib.mfa_gemm_kernel_block_dimensions(self._handle, ctypes.byref(out)))
        return (out[0], out[1], out[2])

    @property
    def threadgroupSize(self) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_gemm_kernel_threadgroup_size(self._handle, ctypes.byref(out)))
        return out.value

    @property
    def threadgroupMemoryAllocation(self) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_gemm_kernel_threadgroup_memory_allocation(self._handle, ctypes.byref(out)))
        return out.value

    def gridSize(self, constants: GEMMFunctionConstantValues) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_gemm_kernel_grid_size(self._handle, ctypes.byref(constants._c), ctypes.byref(out)))
        return out.value

    def launchCount(self, constants: GEMMFunctionConstantValues) -> int:
        out = ctypes.c_uint32()
        _check(_lib.mfa_gemm_kernel_launch_count(self._handle, ctypes.byref(constants._c), ctypes.byref(out)))
        return out.value

    def sourceName(self) -> str:
        return _lib.mfa_gemm_kernel_source_name(self._handle).decode()

    def encode(self, constants: GEMMFunctionConstantValues, buffers: Sequence[int], stream: int = 0) -> None:
        """buffers: device pointers of (A, B, C); stream: cudaStream_t as int (0 = default)."""
        if len(buffers) != MFA_GEMM_BUFFER_COUNT:
            raise MFAError(-2, "GEMM encode takes three buffers: A, B, C.")
        arr = (ctypes.c_void_p * MFA_GEMM_BUFFER_COUNT)(*buffers)
        _check(_lib.mfa_gemm_kernel_encode(self._handle, ctypes.byref(constants._c), ctypes.byref(arr),
                                           ctypes.c_void_p(stream)))


__all__ = [
    "GEMMDescriptor", "GEMMFunctionConstantValues", "GEMMKernelDescriptor", "GEMMKernel",
    "AttentionDescriptor", "AttentionKernelDescriptor", "AttentionKernel", "AttentionKernelType",
    "AttentionOperand", "GEMMOperandPrecision", "FunctionConstantValues", "Backend", "MFAError",
    "library_path", "version", "setParameterTable", "maxExp2FmaQuarters", "hostAlloc", "hostFree", "bindThreadToDevice", "releaseDeviceResources",
]
