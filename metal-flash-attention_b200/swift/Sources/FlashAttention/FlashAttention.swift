//
//  FlashAttention.swift -- drop-in Swift surface over the B200 C ABI.
//
//  Same public names, fields and failure behaviour as the reference package
//  (Sources/FlashAttention/Attention/*.swift, Sources/FlashAttention/GEMM/*.swift), minus everything
//  Metal-specific:
//    * `createSource()` is replaced by `encode(...)`: the kernels are ahead-of-time compiled CUDA, so
//      the compile + bind + dispatch the reference leaves to its caller happens behind the C ABI.
//    * `setFunctionConstants(_:)` fills a plain struct instead of MTLFunctionConstantValues.
//  Where the reference calls fatalError(...), so does this shim (with the C ABI's message).
//
import CMFAB200

/// GEMMOperandPrecision.swift:33-61 (raw values are shared with the C ABI).
public enum GEMMOperandPrecision: UInt16 {
  case FP32 = 0
  case FP16 = 1
  case BF16 = 2
  public var size: Int { self == .FP32 ? 4 : 2 }
  public var name: String { String(cString: mfa_precision_name(mfa_precision_t(UInt32(rawValue)))) }
}

/// AttentionKernelType.swift:8-23
public enum AttentionKernelType: UInt32 {
  case forward = 0
  case backwardQuery = 1
  case backwardKeyValue = 2
}

/// AttentionOperand.swift:8-72; raw values 0...9 are the buffer bindings.
public enum AttentionOperand: UInt32, Hashable, CustomStringConvertible {
  case Q = 0, K, V, O, L, D, dO, dV, dK, dQ, S, P, dP, dS
  public var description: String { String(cString: mfa_operand_name(mfa_operand_t(rawValue))) }
  public var bufferBinding: UInt8? {
    let binding = mfa_operand_buffer_binding(mfa_operand_t(rawValue))
    return binding < 0 ? nil : UInt8(binding)
  }
}

@inline(__always) private func check(_ status: Int32) {
  if status != 0 { fatalError(String(cString: mfa_last_error())) }
}

/// AttentionDescriptor.swift:10-27
public struct AttentionDescriptor {
  public var lowPrecisionInputs: Bool = false
  public var lowPrecisionIntermediates: Bool = false
  public var matrixDimensions: (row: UInt32, column: UInt32, head: UInt16)?
  public var transposeState: (Q: Bool, K: Bool, V: Bool, O: Bool)?
  /// B200 extension: BF16 Q/K/V/dO in memory (nil = the reference's FP16 policy).
  public var inputPrecisionOverride: GEMMOperandPrecision?
  /// B200 extension: number of independent single-head problems stored back to back.
  public var batchCount: UInt32 = 1

  public init() {}

  var c: mfa_attention_descriptor_t {
    var d = mfa_attention_descriptor_t()
    mfa_attention_descriptor_init(&d)
    d.low_precision_inputs = lowPrecisionInputs ? 1 : 0
    d.low_precision_intermediates = lowPrecisionIntermediates ? 1 : 0
    if let m = matrixDimensions {
      d.has_matrix_dimensions = 1
      d.row = m.row; d.column = m.column; d.head = m.head
    }
    if let t = transposeState {
      d.has_transpose_state = 1
      d.transpose_Q = t.Q ? 1 : 0; d.transpose_K = t.K ? 1 : 0
      d.transpose_V = t.V ? 1 : 0; d.transpose_O = t.O ? 1 : 0
    }
    d.input_precision_override = UInt8(inputPrecisionOverride?.rawValue ?? 0)
    d.batch_count = batchCount
    return d
  }

  /// AttentionDescriptor.swift:33-130
  public func kernelDescriptor(type: AttentionKernelType) -> AttentionKernelDescriptor {
    var descriptor = c
    var output = AttentionKernelDescriptor()
    check(mfa_attention_descriptor_kernel_descriptor(&descriptor, mfa_kernel_type_t(type.rawValue), &output.c))
    return output
  }

  /// AttentionDescriptor+Precisions.swift:10-146
  public var memoryPrecisions: [AttentionOperand: GEMMOperandPrecision] {
    var descriptor = c
    var output: [AttentionOperand: GEMMOperandPrecision] = [:]
    for raw in UInt32(0)..<UInt32(MFA_BUFFER_COUNT) {
      var precision = mfa_precision_t(0)
      check(mfa_attention_descriptor_memory_precision(&descriptor, mfa_operand_t(raw), &precision))
      output[AttentionOperand(rawValue: raw)!] = GEMMOperandPrecision(rawValue: UInt16(precision.rawValue))!
    }
    return output
  }

  /// AttentionDescriptor+Precisions.swift:149-215.  P and dS read as the 16-bit input type whenever the tensor-core
  /// family serves the descriptor (they are MMA operands there) -- see `registerPrecisions` of the kernel descriptor
  /// for the per-kernel view.
  public var registerPrecisions: [AttentionOperand: GEMMOperandPrecision] {
    var descriptor = c
    var output: [AttentionOperand: GEMMOperandPrecision] = [:]
    for raw in UInt32(0)..<UInt32(MFA_OPERAND_COUNT) {
      var precision = mfa_precision_t(0)
      check(mfa_attention_descriptor_register_precision(&descriptor, mfa_operand_t(raw), &precision))
      output[AttentionOperand(rawValue: raw)!] = GEMMOperandPrecision(rawValue: UInt16(precision.rawValue))!
    }
    return output
  }

  /// AttentionDescriptor.swift:139-148 (R at index 0, C at index 1).
  public func setFunctionConstants(_ constants: inout mfa_function_constants_t) {
    var descriptor = c
    check(mfa_attention_descriptor_set_function_constants(&descriptor, &constants))
  }

  /// The B200 parameter table this descriptor reads for `type` (AttentionDescriptor+Parameters.swift:106-285 format).
  public func parameterFile(type: AttentionKernelType) -> String {
    var descriptor = c
    return String(cString: mfa_attention_descriptor_parameter_file(&descriptor, mfa_kernel_type_t(type.rawValue)))
  }

  /// Elements of `operand`'s buffer (all `batchCount` problems).
  public func operandElements(_ operand: AttentionOperand) -> Int {
    var descriptor = c
    var count = 0
    check(mfa_attention_descriptor_operand_elements(&descriptor, mfa_operand_t(operand.rawValue), &count))
    return count
  }

  /// End-to-end call on HOST pointers (mfa_attention_run_host): H2D -> the selected kernels in the reference's order
  /// forward -> backwardQuery -> backwardKeyValue (SquareAttentionTest.swift:355-368) -> D2H, synchronous.
  public func runHost(types: [AttentionKernelType],
                      hostBuffers: [AttentionOperand: UnsafeMutableRawPointer],
                      device: Int32 = 0) {
    var descriptor = c
    var mask: UInt32 = 0
    for type in types { mask |= 1 << type.rawValue }
    var table = [UnsafeMutableRawPointer?](repeating: nil, count: Int(MFA_BUFFER_COUNT))
    for (operand, pointer) in hostBuffers {
      guard let binding = operand.bufferBinding else { fatalError("Operand \(operand) has no buffer binding.") }
      table[Int(binding)] = pointer
    }
    check(mfa_attention_run_host(&descriptor, mask, &table, device))
  }
}

/// Page-locked host buffers on the GPU's NUMA node for `AttentionDescriptor.runHost` (B200 extension).
public enum HostMemory {
  /// `upload`: write-combined pages for buffers the host only writes and the GPU reads (Q, K, V, dO).
  public static func allocate(byteCount: Int, device: Int32 = 0, upload: Bool = false) -> UnsafeMutableRawPointer {
    var pointer: UnsafeMutableRawPointer?
    check(upload ? mfa_host_alloc_upload(byteCount, device, &pointer) : mfa_host_alloc(byteCount, device, &pointer))
    return pointer!
  }
  public static func free(_ pointer: UnsafeMutableRawPointer) { check(mfa_host_free(pointer)) }
  /// Pins the calling thread to the CPUs of the GPU's NUMA node; returns the node (-1: none reported).
  @discardableResult public static func bindThread(toDevice device: Int32) -> Int32 {
    var node: Int32 = -1
    check(mfa_host_bind_thread_to_device(device, &node))
    return node
  }
  /// Frees the library's scratch and workspaces on `device`.
  public static func releaseResources(device: Int32) { check(mfa_release_device_resources(device)) }
}

/// Which kernel family serves a descriptor (B200 extension; the reference has one family).
public enum AttentionBackend: UInt8 {
  case simtFP32 = 0
  case tcgen05 = 1
}

/// AttentionKernelDescriptor.swift:7-48 -- a plain, editable value.  Every field of the reference's struct is here,
/// readable and settable with the same types (optionals start as nil, dictionaries empty); storage is the C struct.
public struct AttentionKernelDescriptor {
  public var c = mfa_attention_kernel_descriptor_t()
  public init() { mfa_attention_kernel_descriptor_init(&c) }

  /// :8  blockDimensions
  public var blockDimensions: (parallelization: UInt16, traversal: UInt16, head: UInt16)? {
    get { c.has_block_dimensions == 0 ? nil : (c.block_parallelization, c.block_traversal, c.block_head) }
    set {
      c.has_block_dimensions = newValue == nil ? 0 : 1
      c.block_parallelization = newValue?.parallelization ?? 0
      c.block_traversal = newValue?.traversal ?? 0
      c.block_head = newValue?.head ?? 0
    }
  }

  /// :11  cacheState -- whether each operand stays resident on chip for the whole traversal
  public var cacheState: [AttentionOperand: Bool] {
    get {
      var output: [AttentionOperand: Bool] = [:]
      for raw in UInt32(0)..<UInt32(MFA_OPERAND_COUNT) where (c.cache_state_valid_mask >> UInt16(raw)) & 1 == 1 {
        output[AttentionOperand(rawValue: raw)!] = (c.cache_state_mask >> UInt16(raw)) & 1 == 1
      }
      return output
    }
    set {
      c.cache_state_valid_mask = 0
      c.cache_state_mask = 0
      for (operand, cached) in newValue {
        c.cache_state_valid_mask |= 1 << UInt16(operand.rawValue)
        if cached { c.cache_state_mask |= 1 << UInt16(operand.rawValue) }
      }
    }
  }

  /// :14  headDimension
  public var headDimension: UInt16? {
    get { c.has_head_dimension == 0 ? nil : c.head_dimension }
    set {
      c.has_head_dimension = newValue == nil ? 0 : 1
      c.head_dimension = newValue ?? 0
    }
  }

  private static func precisions(_ tuple: inout mfa_attention_kernel_descriptor_t,
                                 register: Bool) -> [AttentionOperand: GEMMOperandPrecision] {
    var output: [AttentionOperand: GEMMOperandPrecision] = [:]
    for raw in UInt32(0)..<UInt32(MFA_OPERAND_COUNT) {
      let value = mfa_attention_kernel_descriptor_get_precision(&tuple, mfa_operand_t(raw), register ? 1 : 0)
      if value >= 0 { output[AttentionOperand(rawValue: raw)!] = GEMMOperandPrecision(rawValue: UInt16(value))! }
    }
    return output
  }
  private static func setPrecisions(_ tuple: inout mfa_attention_kernel_descriptor_t, register: Bool,
                                    _ values: [AttentionOperand: GEMMOperandPrecision]) {
    for raw in UInt32(0)..<UInt32(MFA_OPERAND_COUNT) {
      let value = values[AttentionOperand(rawValue: raw)!].map { Int32($0.rawValue) } ?? -1
      mfa_attention_kernel_descriptor_set_precision(&tuple, mfa_operand_t(raw), register ? 1 : 0, value)
    }
  }

  /// :17  memoryPrecisions
  public var memoryPrecisions: [AttentionOperand: GEMMOperandPrecision] {
    get { var copy = c; return Self.precisions(&copy, register: false) }
    set { Self.setPrecisions(&c, register: false, newValue) }
  }
  /// :19  registerPrecisions
  public var registerPrecisions: [AttentionOperand: GEMMOperandPrecision] {
    get { var copy = c; return Self.precisions(&copy, register: true) }
    set { Self.setPrecisions(&c, register: true, newValue) }
  }

  /// :22  preferAsyncCache ("async" == TMA bulk-tensor copies on B200)
  public var preferAsyncCache: Bool? {
    get { c.prefer_async_cache == 0xFF ? nil : c.prefer_async_cache != 0 }
    set { c.prefer_async_cache = newValue.map { $0 ? 1 : 0 } ?? 0xFF }
  }
  /// :25  preferAsyncLoad
  public var preferAsyncLoad: Bool? {
    get { c.prefer_async_load == 0xFF ? nil : c.prefer_async_load != 0 }
    set { c.prefer_async_load = newValue.map { $0 ? 1 : 0 } ?? 0xFF }
  }

  /// :42  transposeState -- per operand; derivatives follow their forward operand (AttentionDescriptor.swift:96-111)
  public var transposeState: [AttentionOperand: Bool] {
    get {
      var output: [AttentionOperand: Bool] = [:]
      for raw in UInt32(0)..<UInt32(MFA_OPERAND_COUNT) where (c.transpose_state_valid_mask >> UInt16(raw)) & 1 == 1 {
        output[AttentionOperand(rawValue: raw)!] = (c.transpose_state_mask >> UInt16(raw)) & 1 == 1
      }
      return output
    }
    set {
      c.transpose_state_valid_mask = 0
      c.transpose_state_mask = 0
      for (operand, transposed) in newValue {
        c.transpose_state_valid_mask |= 1 << UInt16(operand.rawValue)
        if transposed { c.transpose_state_mask |= 1 << UInt16(operand.rawValue) }
      }
    }
  }

  /// :45  type
  public var type: AttentionKernelType? {
    get { c.type == 0xFF ? nil : AttentionKernelType(rawValue: UInt32(c.type)) }
    set { c.type = newValue.map { UInt8($0.rawValue) } ?? 0xFF }
  }

  /// B200 extension: the kernel family `AttentionDescriptor.kernelDescriptor(type:)` selected.
  public var backend: AttentionBackend {
    get { AttentionBackend(rawValue: c.backend) ?? .simtFP32 }
    set { c.backend = newValue.rawValue }
  }
  /// B200 extension: tuning columns of the parameter-table row.  Of every 4 element pairs of P, how many take exp2 on
  /// the FMA pipe (selects the kernel instantiation); small-grid split policy (minimum blocks per range, 0 = never;
  /// maximum ranges).
  public var exp2FmaQuarters: UInt8 {
    get { c.exp2_fma_quarters }
    set { c.exp2_fma_quarters = newValue }
  }
  public var splitPolicy: (minimumBlocks: UInt8, maximumSplits: UInt8) {
    get { (c.split_min_blocks, c.split_max) }
    set { c.split_min_blocks = newValue.minimumBlocks; c.split_max = newValue.maximumSplits }
  }
}

/// The parameter tables are data (AttentionDescriptor+Parameters.swift:106-285): replace the tensor-core family's table
/// of `type` at run time (`nil` restores the built-in one).
public func setParameterTable(type: AttentionKernelType, text: String?, transposed: Bool = false) {
  if let text = text {
    text.withCString { check(mfa_set_parameter_table(mfa_kernel_type_t(type.rawValue), transposed ? 1 : 0, $0)) }
  } else {
    check(mfa_set_parameter_table(mfa_kernel_type_t(type.rawValue), transposed ? 1 : 0, nil))
  }
}

/// AttentionKernel.swift:11-50, 268-363
public final class AttentionKernel {
  let handle: OpaquePointer
  let owned: Bool

  public init(descriptor: AttentionKernelDescriptor) {
    var kd = descriptor.c
    var out: OpaquePointer?
    check(mfa_attention_kernel_create(&kd, &out))
    handle = out!
    owned = true
  }
  /// Library-owned kernel object from the descriptor-keyed cache -- the analogue of
  /// `GEMMKernel.pipelineCache[descriptor]` (GEMMDescriptor+PipelineCache.swift:16-36).
  public init(cached descriptor: AttentionDescriptor, type: AttentionKernelType) {
    var d = descriptor.c
    var out: OpaquePointer?
    check(mfa_attention_kernel_cache_fetch(&d, mfa_kernel_type_t(type.rawValue), &out))
    handle = out!
    owned = false
  }
  deinit { if owned { mfa_attention_kernel_destroy(handle) } }

  public var blockDimensions: (parallelization: UInt16, traversal: UInt16, head: UInt16) {
    var out: (UInt16, UInt16, UInt16) = (0, 0, 0)
    withUnsafeMutablePointer(to: &out) {
      $0.withMemoryRebound(to: UInt16.self, capacity: 3) { check(mfa_attention_kernel_block_dimensions(handle, $0)) }
    }
    return out
  }
  public var threadgroupSize: UInt32 {
    var out: UInt32 = 0
    check(mfa_attention_kernel_threadgroup_size(handle, &out))
    return out
  }
  public var threadgroupMemoryAllocation: UInt32 {
    var out: UInt32 = 0
    check(mfa_attention_kernel_threadgroup_memory_allocation(handle, &out))
    return out
  }

  /// Thread blocks along the parallelization dimension (R for forward / backwardQuery, C for backwardKeyValue) times
  /// the batch: what the reference's caller computes for dispatchThreadgroups (SquareAttentionTest.swift:328-339).
  public func gridSize(constants: mfa_function_constants_t) -> UInt32 {
    var constants = constants
    var out: UInt32 = 0
    check(mfa_attention_kernel_grid_size(handle, &constants, &out))
    return out
  }
  /// CUDA kernels one `encode` launches (2 only when a small grid is split and a merge kernel follows).
  public func launchCount(constants: mfa_function_constants_t) -> UInt32 {
    var constants = constants
    var out: UInt32 = 0
    check(mfa_attention_kernel_launch_count(handle, &constants, &out))
    return out
  }
  /// Stands in for `createSource()` (AttentionKernel+Source.swift:11-55): the name of the ahead-of-time compiled kernel.
  public var sourceName: String { String(cString: mfa_attention_kernel_source_name(handle)) }

  /// What the reference's callers do by hand around `createSource()` (SquareAttentionTest.swift:240-372):
  /// `buffers[binding]` are DEVICE pointers at AttentionOperand.bufferBinding; `stream` is a cudaStream_t.
  public func encode(constants: mfa_function_constants_t,
                     buffers: [AttentionOperand: UnsafeMutableRawPointer],
                     stream: UnsafeMutableRawPointer? = nil) {
    var table = [UnsafeMutableRawPointer?](repeating: nil, count: Int(MFA_BUFFER_COUNT))
    for (operand, pointer) in buffers {
      guard let binding = operand.bufferBinding else { fatalError("Operand \(operand) has no buffer binding.") }
      table[Int(binding)] = pointer
    }
    var constants = constants
    check(mfa_attention_kernel_encode(handle, &constants, &table, stream))
  }
}

// MARK: - GEMM (Sources/FlashAttention/GEMM/): C = A . B, or C += A . B with loadPreviousC

/// GEMMDescriptor.swift:10-44
public struct GEMMDescriptor: Hashable {
  /// B200 extension beyond the block-size heuristic: N > 1 runs N problems stored back to back.
  public var batchDimension: Int = 1
  public var leadingDimensions: (A: UInt32, B: UInt32, C: UInt32)?
  public var loadPreviousC: Bool = false
  public var matrixDimensions: (M: UInt32, N: UInt32, K: UInt32)?
  public var memoryPrecisions: (A: GEMMOperandPrecision, B: GEMMOperandPrecision, C: GEMMOperandPrecision)?
  public var transposeState: (A: Bool, B: Bool)?

  public init() {}

  var c: mfa_gemm_descriptor_t {
    var d = mfa_gemm_descriptor_t()
    mfa_gemm_descriptor_init(&d)
    d.batch_dimension = UInt32(batchDimension)
    if let l = leadingDimensions {
      d.has_leading_dimensions = 1
      d.leading_dimensions = (l.A, l.B, l.C)
    }
    d.load_previous_C = loadPreviousC ? 1 : 0
    if let m = matrixDimensions {
      d.has_matrix_dimensions = 1
      d.M = m.M; d.N = m.N; d.K = m.K
    }
    if let p = memoryPrecisions {
      d.has_memory_precisions = 1
      d.memory_precisions = (UInt8(p.A.rawValue), UInt8(p.B.rawValue), UInt8(p.C.rawValue))
    }
    if let t = transposeState {
      d.has_transpose_state = 1
      d.transpose_A = t.A ? 1 : 0; d.transpose_B = t.B ? 1 : 0
    }
    return d
  }

  /// GEMMDescriptor.swift:327-380: M, N, K, the leading dimensions (chooseLeadingDimension's defaults when nil),
  /// loadPreviousC and the batch, into a plain struct instead of MTLFunctionConstantValues.
  public func setFunctionConstants(_ constants: inout mfa_gemm_function_constants_t) {
    var d = c
    check(mfa_gemm_descriptor_set_function_constants(&d, &constants))
  }

  // Equal when GEMMKey (GEMMDescriptor.swift:49-90) is: the C struct is compared field by field.
  public static func == (lhs: GEMMDescriptor, rhs: GEMMDescriptor) -> Bool {
    let l = lhs.c, r = rhs.c
    return withUnsafeBytes(of: l) { a in withUnsafeBytes(of: r) { b in a.elementsEqual(b) } }
  }
  public func hash(into hasher: inout Hasher) {
    withUnsafeBytes(of: c) { hasher.combine(bytes: $0) }
  }
}

/// GEMMKernelDescriptor.swift:21-181 -- a plain, editable value; storage is the C struct.
public struct GEMMKernelDescriptor {
  public var c = mfa_gemm_kernel_descriptor_t()
  public init() { mfa_gemm_kernel_descriptor_init(&c) }
  /// GEMMDescriptor.swift:106-234, with this library's heuristic: the tcgen05 family when A and B are both FP16 or
  /// both BF16, the SIMT FP32 family otherwise; register precisions (A, B as in memory, C FP32).
  public init(descriptor: GEMMDescriptor) {
    var d = descriptor.c
    check(mfa_gemm_descriptor_kernel_descriptor(&d, &c))
  }

  public var blockDimensions: (M: UInt16, N: UInt16, K: UInt16)? {
    get { c.has_block_dimensions != 0 ? c.block_dimensions : nil }
    set {
      c.has_block_dimensions = newValue == nil ? 0 : 1
      if let v = newValue { c.block_dimensions = (v.M, v.N, v.K) }
    }
  }
  public var leadingBlockDimensions: (A: UInt16, B: UInt16, C: UInt16)? {
    get { c.has_leading_block_dimensions != 0 ? c.leading_block_dimensions : nil }
    set {
      c.has_leading_block_dimensions = newValue == nil ? 0 : 1
      if let v = newValue { c.leading_block_dimensions = (v.A, v.B, v.C) }
    }
  }
  private static func precisions(_ t: (UInt8, UInt8, UInt8))
    -> (A: GEMMOperandPrecision, B: GEMMOperandPrecision, C: GEMMOperandPrecision) {
    (GEMMOperandPrecision(rawValue: UInt16(t.0))!, GEMMOperandPrecision(rawValue: UInt16(t.1))!,
     GEMMOperandPrecision(rawValue: UInt16(t.2))!)
  }
  public var memoryPrecisions: (A: GEMMOperandPrecision, B: GEMMOperandPrecision, C: GEMMOperandPrecision)? {
    get { c.has_memory_precisions != 0 ? Self.precisions(c.memory_precisions) : nil }
    set {
      c.has_memory_precisions = newValue == nil ? 0 : 1
      if let v = newValue { c.memory_precisions = (UInt8(v.A.rawValue), UInt8(v.B.rawValue), UInt8(v.C.rawValue)) }
    }
  }
  public var registerPrecisions: (A: GEMMOperandPrecision, B: GEMMOperandPrecision, C: GEMMOperandPrecision)? {
    get { c.has_register_precisions != 0 ? Self.precisions(c.register_precisions) : nil }
    set {
      c.has_register_precisions = newValue == nil ? 0 : 1
      if let v = newValue { c.register_precisions = (UInt8(v.A.rawValue), UInt8(v.B.rawValue), UInt8(v.C.rawValue)) }
    }
  }
  public var preferAsyncLoad: Bool {
    get { c.prefer_async_load != 0 }
    set { c.prefer_async_load = newValue ? 1 : 0 }
  }
  public var preferAsyncStore: Bool? {
    get { c.prefer_async_store == 0xFF ? nil : c.prefer_async_store != 0 }
    set { c.prefer_async_store = newValue.map { $0 ? 1 : 0 } ?? 0xFF }
  }
  public var splits: (M: UInt16, N: UInt16)? {
    get { c.has_splits != 0 ? c.splits : nil }
    set {
      c.has_splits = newValue == nil ? 0 : 1
      if let v = newValue { c.splits = (v.M, v.N) }
    }
  }
  public var transposeState: (A: Bool, B: Bool)? {
    get { c.has_transpose_state != 0 ? (c.transpose_A != 0, c.transpose_B != 0) : nil }
    set {
      c.has_transpose_state = newValue == nil ? 0 : 1
      if let v = newValue { c.transpose_A = v.A ? 1 : 0; c.transpose_B = v.B ? 1 : 0 }
    }
  }
  /// B200 extension: which sm_100a kernel family the heuristic picked.
  public var backend: AttentionBackend {
    get { AttentionBackend(rawValue: c.backend)! }
    set { c.backend = newValue.rawValue }
  }
}

/// GEMMKernel.swift:10-270
public final class GEMMKernel {
  let handle: OpaquePointer
  let owned: Bool

  public init(descriptor: GEMMKernelDescriptor) {
    var kd = descriptor.c
    var out: OpaquePointer?
    check(mfa_gemm_kernel_create(&kd, &out))
    handle = out!
    owned = true
  }
  init(cached descriptor: GEMMDescriptor) {
    var d = descriptor.c
    var out: OpaquePointer?
    check(mfa_gemm_kernel_cache_fetch(&d, &out))
    handle = out!
    owned = false
  }
  deinit { if owned { mfa_gemm_kernel_destroy(handle) } }

  /// GEMMDescriptor+PipelineCache.swift:24-36: creates the descriptor's kernel object once.  The cache key is the
  /// precisions and transposes; M, N, K, leading dimensions, loadPreviousC and the batch are launch constants.
  public static func register(descriptor: GEMMDescriptor) { _ = GEMMKernel(cached: descriptor) }
  /// `pipelineCache[descriptor]`: the library-owned kernel object (registered on first use).
  public static func cached(descriptor: GEMMDescriptor) -> GEMMKernel { GEMMKernel(cached: descriptor) }
  public static var cacheSize: Int { Int(mfa_gemm_kernel_cache_size()) }

  public var blockDimensions: (M: UInt16, N: UInt16, K: UInt16) {
    var out: (UInt16, UInt16, UInt16) = (0, 0, 0)
    withUnsafeMutablePointer(to: &out) {
      $0.withMemoryRebound(to: UInt16.self, capacity: 3) { check(mfa_gemm_kernel_block_dimensions(handle, $0)) }
    }
    return out
  }
  public var threadgroupSize: UInt32 {
    var out: UInt32 = 0
    check(mfa_gemm_kernel_threadgroup_size(handle, &out))
    return out
  }
  public var threadgroupMemoryAllocation: UInt32 {
    var out: UInt32 = 0
    check(mfa_gemm_kernel_threadgroup_memory_allocation(handle, &out))
    return out
  }
  /// Output tiles: ceil(N / block N) * ceil(M / block M) * batch (AdversarialShapeTest.swift:155-158).
  public func gridSize(constants: mfa_gemm_function_constants_t) -> UInt32 {
    var constants = constants
    var out: UInt32 = 0
    check(mfa_gemm_kernel_grid_size(handle, &constants, &out))
    return out
  }
  /// CUDA kernels one `encode` launches: 1, plus a staging copy per 16-bit operand TMA cannot address in place.
  public func launchCount(constants: mfa_gemm_function_constants_t) -> UInt32 {
    var constants = constants
    var out: UInt32 = 0
    check(mfa_gemm_kernel_launch_count(handle, &constants, &out))
    return out
  }
  /// Stands in for `createSource()`: the name of the ahead-of-time compiled kernel.
  public var sourceName: String { String(cString: mfa_gemm_kernel_source_name(handle)) }

  /// Binds A, B, C (DEVICE pointers, bindings 0, 1, 2 as in GEMMKernel+Source.swift:42-44) and dispatches on `stream`
  /// (a cudaStream_t): what AdversarialShapeTest.swift:140-169 does by hand around the Metal pipeline.
  public func encode(constants: mfa_gemm_function_constants_t,
                     A: UnsafeRawPointer, B: UnsafeRawPointer, C: UnsafeMutableRawPointer,
                     stream: UnsafeMutableRawPointer? = nil) {
    var table: [UnsafeMutableRawPointer?] = [UnsafeMutableRawPointer(mutating: A), UnsafeMutableRawPointer(mutating: B), C]
    var constants = constants
    check(mfa_gemm_kernel_encode(handle, &constants, &table, stream))
  }
}
