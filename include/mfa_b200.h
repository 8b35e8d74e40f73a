/*
 * mfa_b200.h -- C ABI of the B200-native FlashAttention hot path that stands in for
 * philipturner/metal-flash-attention's attention path.
 *
 * The reference's boundary is a set of Swift value types that *describe* a kernel and hand the
 * caller a Metal source string plus launch geometry; the caller compiles, binds ten buffers and
 * dispatches (Tests/FlashAttentionTests/Attention/SquareAttentionTest.swift:226-380).  This
 * header keeps that shape 1:1 (same names, same fields, same validation rules) and moves the
 * part the reference leaves to its caller -- compile + bind + dispatch -- behind
 * mfa_attention_kernel_encode(), because on B200 the kernels are pre-compiled sm_100a CUDA.
 *
 * Conventions
 *   - Plain C: pointers, sizes, enums with fixed raw values.  No torch / C++ types.
 *   - Every function returns MFA_SUCCESS (0) or a negative mfa_status_t; the message for the
 *     calling thread is available from mfa_last_error().  Where the reference calls
 *     fatalError() the ABI returns an error with the reference's message text (a C ABI must not
 *     abort its host); the Swift / C++ / Python mirrors turn that back into a trap/exception.
 *   - The library never owns caller buffers.  Device entry points take device pointers and a
 *     cudaStream_t (as void*) and are asynchronous on that stream.  The *_host entry point takes
 *     host pointers and performs H2D -> kernels -> D2H itself.
 *   - A kernel handle is immutable after creation and may be encoded concurrently from several
 *     threads / streams.
 *   - There is NO CPU fallback: if no sm_100 device / driver is present, encode fails loudly
 *     with MFA_ERROR_NO_DEVICE.
 *
 * Reference citations use R/ = /root/reference/Sources/FlashAttention/.
 */
#ifndef MFA_B200_H
#define MFA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MFA_API __attribute__((visibility("default")))
#else
#define MFA_API
#endif

/* ------------------------------------------------------------------------------------------ */
/* Status                                                                                      */
/* ------------------------------------------------------------------------------------------ */
typedef enum mfa_status {
  MFA_SUCCESS = 0,
  MFA_ERROR_INCOMPLETE_DESCRIPTOR = -1, /* "Descriptor was incomplete."  R/Attention/AttentionDescriptor/AttentionDescriptor.swift:89-91, AttentionKernel.swift:28-34 */
  MFA_ERROR_INVALID_ARGUMENT = -2,      /* NULL pointer, enum out of range, operand without a buffer */
  MFA_ERROR_UNEXPECTED_OPERAND = -3,    /* "Unexpected operand: X"  AttentionDescriptor.swift:69-74 */
  MFA_ERROR_INVALID_PRECISIONS = -4,    /* "Invalid precisions."  AttentionKernel.swift:90-105 */
  MFA_ERROR_UNSUPPORTED = -5,           /* shape outside what the sm_100a kernels cover (e.g. head > 512) */
  MFA_ERROR_NO_DEVICE = -6,             /* no CUDA device / not sm_100 -- never falls back to a CPU path */
  MFA_ERROR_CUDA = -7                   /* a CUDA runtime / driver call failed; message has the detail */
} mfa_status_t;

/** Thread-local, NUL-terminated description of the last error on the calling thread. */
MFA_API const char *mfa_last_error(void);

/** Library version / build info ("mfa_b200 x.y sm_100a"). */
MFA_API const char *mfa_version(void);

/* ------------------------------------------------------------------------------------------ */
/* Enumerations (raw values are part of the ABI)                                               */
/* ------------------------------------------------------------------------------------------ */

/** = GEMMOperandPrecision raw values.  R/GEMM/GEMMOperandPrecision.swift:33-37 */
typedef enum mfa_precision { MFA_FP32 = 0, MFA_FP16 = 1, MFA_BF16 = 2 } mfa_precision_t;

/** Size of one scalar in bytes.  GEMMOperandPrecision.size, R/GEMM/GEMMOperandPrecision.swift:51-60 */
MFA_API int mfa_precision_size(mfa_precision_t precision);
/** "float" / "half" / "bfloat".  GEMMOperandPrecision.name, :39-48 */
MFA_API const char *mfa_precision_name(mfa_precision_t precision);

/** = AttentionKernelType.  R/Attention/AttentionKernelType.swift:8-23 */
typedef enum mfa_kernel_type {
  MFA_FORWARD = 0,           /* computes O and L */
  MFA_BACKWARD_QUERY = 1,    /* computes D and dQ; depends on L */
  MFA_BACKWARD_KEY_VALUE = 2 /* computes dK and dV; depends on L and D */
} mfa_kernel_type_t;

/** = AttentionOperand.  Values 0..9 ARE the buffer bindings (AttentionOperand.bufferBinding,
 *  R/Attention/AttentionOperand.swift:52-71); S, P, dP, dS are never materialised (binding nil). */
typedef enum mfa_operand {
  MFA_Q = 0, MFA_K = 1, MFA_V = 2, MFA_O = 3,
  MFA_L = 4, MFA_D = 5,
  MFA_dO = 6, MFA_dV = 7, MFA_dK = 8, MFA_dQ = 9,
  MFA_S = 10, MFA_P = 11, MFA_dP = 12, MFA_dS = 13,
  MFA_OPERAND_COUNT = 14
} mfa_operand_t;
#define MFA_BUFFER_COUNT 10

/** "Q", "K", ..., "dQ".  AttentionOperand.description, AttentionOperand.swift:29-50 */
MFA_API const char *mfa_operand_name(mfa_operand_t operand);
/** Buffer slot 0..9, or -1 for S/P/dP/dS.  AttentionOperand.bufferBinding, :52-71 */
MFA_API int mfa_operand_buffer_binding(mfa_operand_t operand);

/* ------------------------------------------------------------------------------------------ */
/* AttentionDescriptor   (R/Attention/AttentionDescriptor/AttentionDescriptor.swift:10-27)     */
/* ------------------------------------------------------------------------------------------ */
typedef struct mfa_attention_descriptor {
  uint8_t low_precision_inputs;        /* lowPrecisionInputs (Q, K, V, dO)            :12 */
  uint8_t low_precision_intermediates; /* lowPrecisionIntermediates (S,P,L,D,dP,dS)   :15 */
  uint8_t has_matrix_dimensions;       /* Swift optional `matrixDimensions != nil`    :20 */
  uint8_t has_transpose_state;         /* Swift optional `transposeState != nil`      :22 */
  uint32_t row;                        /* matrixDimensions.row    (output sequence length R) */
  uint32_t column;                     /* matrixDimensions.column (input sequence length C)  */
  uint16_t head;                       /* matrixDimensions.head   (head dimension D)         */
  uint8_t transpose_Q, transpose_K, transpose_V, transpose_O; /* transposeState :22 */
  /* ---- B200 extensions; all-zero reproduces the reference exactly ---- */
  uint8_t input_precision_override;    /* 0: reference policy (Q,K,V FP16 and dO BF16 when lowPrecisionInputs,
                                          AttentionDescriptor+Precisions.swift:13-23);
                                          MFA_BF16 (2): Q,K,V,dO are all BF16 in memory (north_star asks for bf16);
                                          MFA_FP16 (1): Q,K,V,dO are all FP16.
                                          Only meaningful with low_precision_inputs.  All three variants run on the
                                          tensor-core kernels (with the reference policy the backward kernels rewrite
                                          the staged BF16 dO tiles as FP16 on chip: tcgen05 kind::f16 cannot mix
                                          FP16 and BF16 operands in one MMA). */
  uint8_t reserved0;
  uint32_t batch_count;                /* 0 or 1: single head (reference). N > 1: N independent
                                          single-head problems, each operand stored back to back
                                          (operand i of problem b starts at b * elements(i)). */
} mfa_attention_descriptor_t;

/** AttentionDescriptor.init(): all false / nil / zero. */
MFA_API void mfa_attention_descriptor_init(mfa_attention_descriptor_t *descriptor);

/** descriptor.memoryPrecisions[operand]   (AttentionDescriptor+Precisions.swift:10-146).
 *  Operands without a buffer (S,P,dP,dS) -> MFA_ERROR_INVALID_ARGUMENT. */
MFA_API int mfa_attention_descriptor_memory_precision(const mfa_attention_descriptor_t *descriptor,
                                                      mfa_operand_t operand, mfa_precision_t *out);
/** descriptor.registerPrecisions[operand] (AttentionDescriptor+Precisions.swift:149-215), i.e. the
 *  precision the operand has while it is an MMA operand / accumulator on chip. */
MFA_API int mfa_attention_descriptor_register_precision(const mfa_attention_descriptor_t *descriptor,
                                                        mfa_operand_t operand, mfa_precision_t *out);

/* ------------------------------------------------------------------------------------------ */
/* AttentionKernelDescriptor   (R/Attention/AttentionKernelDescriptor.swift:7-48)              */
/* ------------------------------------------------------------------------------------------ */
typedef enum mfa_backend {
  MFA_BACKEND_SIMT_FP32 = 0, /* CUDA-core FP32 FMA kernels: any R, C, D <= 512, any transposes/precisions */
  MFA_BACKEND_TCGEN05 = 1    /* TMA + tcgen05.mma + TMEM kernels: 16-bit inputs, D % 8 == 0; forward D <= 256 (transposed
                                operands too, where the transposed row pitch is a multiple of 16 bytes), backward D <= 128
                                row-major */
} mfa_backend_t;

typedef struct mfa_attention_kernel_descriptor {
  /* blockDimensions (parallelization, traversal, head)                               :8-9   */
  uint8_t has_block_dimensions;
  uint16_t block_parallelization, block_traversal, block_head;
  /* cacheState: bit i set <=> operand i is kept resident on chip for the whole traversal
     (registers on Apple GPUs; SMEM / TMEM / registers on B200).                      :12    */
  uint16_t cache_state_valid_mask; /* which operands have an entry at all */
  uint16_t cache_state_mask;
  /* headDimension                                                                    :15    */
  uint8_t has_head_dimension;
  uint16_t head_dimension;
  /* memoryPrecisions / registerPrecisions; 0xFF = no entry                           :17,25 */
  uint8_t memory_precisions[MFA_OPERAND_COUNT];
  uint8_t register_precisions[MFA_OPERAND_COUNT];
  /* preferAsyncCache / preferAsyncLoad: 0 false, 1 true, 0xFF nil.  On B200 "async" means the
     TMA (cp.async.bulk.tensor) path; both are true for MFA_BACKEND_TCGEN05.          :20,23 */
  uint8_t prefer_async_cache, prefer_async_load;
  /* transposeState: bit i set <=> operand i is stored [D][seq] (leading dim = seq).   :27-42 */
  uint16_t transpose_state_valid_mask;
  uint16_t transpose_state_mask;
  /* type; 0xFF = nil                                                                 :44    */
  uint8_t type;
  /* ---- B200 extension: which sm_100a kernel family the heuristic picked ---- */
  uint8_t backend; /* mfa_backend_t */
  /* ---- B200 extension: the tuning columns of the parameter-table row (tcgen05 family).  Like blockDimensions they
     are plain data the caller may edit before AttentionKernel(descriptor:); kernel creation accepts every value that has
     a compiled instantiation (exp2_fma_quarters <= mfa_max_exp2_fma_quarters(type)) and rejects the rest. ---- */
  uint8_t exp2_fma_quarters; /* of every 4 element pairs of P, how many take exp2 on the FMA pipe (Cody-Waite +
                                polynomial) instead of the MUFU pipe: selects the kernel instantiation */
  uint8_t split_min_blocks;  /* small grids: a traversal range handed to one CTA has at least this many 128-key (or
                                128-query) blocks; 0 = never split */
  uint8_t split_max;         /* small grids: at most this many ranges per tile (forward <= 16, backward <= 8) */
} mfa_attention_kernel_descriptor_t;

/** AttentionKernelDescriptor.init(): everything nil / empty. */
MFA_API void mfa_attention_kernel_descriptor_init(mfa_attention_kernel_descriptor_t *kernel_descriptor);

/** Element access to memory_precisions / register_precisions for host languages that import C arrays awkwardly (Swift
 *  sees them as 14-tuples): returns the precision raw value or -1 when unset; set with value < 0 to clear. */
MFA_API int mfa_attention_kernel_descriptor_get_precision(const mfa_attention_kernel_descriptor_t *kernel_descriptor,
                                                          mfa_operand_t operand, int register_file);
MFA_API void mfa_attention_kernel_descriptor_set_precision(mfa_attention_kernel_descriptor_t *kernel_descriptor,
                                                           mfa_operand_t operand, int register_file, int value);

/** descriptor.kernelDescriptor(type:)  (AttentionDescriptor.swift:33-130): looks up the B200
 *  parameter table for (type, precision class), picks the first row with head <= max head
 *  (AttentionDescriptor+Parameters.swift:41-66), clamps the head block to pad8(D) (:41-54),
 *  validates the cached-operand list (:56-86) and mirrors the transposes onto dO/dV/dK/dQ
 *  (:96-111).  Errors: MFA_ERROR_INCOMPLETE_DESCRIPTOR, MFA_ERROR_UNEXPECTED_OPERAND. */
MFA_API int mfa_attention_descriptor_kernel_descriptor(const mfa_attention_descriptor_t *descriptor,
                                                       mfa_kernel_type_t type,
                                                       mfa_attention_kernel_descriptor_t *out);

/** The parameter table text that kernelDescriptor(type:) would parse for this descriptor -- the analogue of
 *  AttentionDescriptor.parameterFile(type:) (AttentionDescriptor+Parameters.swift:13-39).  Rows are the reference's
 *  "| maxD | par | trav | head | cached |" with, for the tcgen05 family, three B200 tuning columns appended:
 *  "| exp2 on the FMA pipe (quarters) | min blocks per split | max splits |".  The returned pointer stays valid until
 *  the table is replaced. */
MFA_API const char *mfa_attention_descriptor_parameter_file(const mfa_attention_descriptor_t *descriptor,
                                                            mfa_kernel_type_t type);

/** The tables are DATA: this replaces the tcgen05-family table of `type` (`transposed` != 0: the table used with transposed operands, i.e. of the
 *  layout-generic kernels) with `text` in the format above; NULL restores the built-in table.  The text is
 *  parsed and validated first (unknown operand names, malformed rows, tuning values without a compiled kernel are
 *  rejected and the current table stays).  Kernels fetched from the descriptor-keyed cache afterwards follow the new
 *  table.  At load time the library also reads the file named by the environment variable MFA_B200_PARAMETER_FILE
 *  (sections "[forward]", "[backwardQuery]", "[backwardKeyValue]", each also as "[....transposed]"; scripts/sweep.py writes
 *  one from measurements on the current GPU).  Not thread-safe against concurrent kernelDescriptor() calls. */
MFA_API int mfa_set_parameter_table(mfa_kernel_type_t type, int transposed, const char *text);
/** Largest exp2_fma_quarters with a compiled instantiation for `type`. */
MFA_API int mfa_max_exp2_fma_quarters(mfa_kernel_type_t type);

/** descriptor.setFunctionConstants(_:)  (AttentionDescriptor.swift:139-148): the two launch-time
 *  constants R (index 0) and C (index 1), plus the batch extension. */
typedef struct mfa_function_constants {
  uint32_t row;         /* R, function constant 0 */
  uint32_t column;      /* C, function constant 1 */
  uint32_t batch_count; /* extension; 0/1 = single head */
} mfa_function_constants_t;
MFA_API int mfa_attention_descriptor_set_function_constants(const mfa_attention_descriptor_t *descriptor,
                                                            mfa_function_constants_t *constants);

/* ------------------------------------------------------------------------------------------ */
/* AttentionKernel   (R/Attention/AttentionKernel/AttentionKernel.swift:11-50, 268-363)        */
/* ------------------------------------------------------------------------------------------ */
typedef struct mfa_attention_kernel mfa_attention_kernel_t; /* opaque */

/** AttentionKernel(descriptor:)  (:27-50).  Incomplete descriptor -> MFA_ERROR_INCOMPLETE_DESCRIPTOR;
 *  illegal memory/register precision pairs (:81-139) -> MFA_ERROR_INVALID_PRECISIONS. */
MFA_API int mfa_attention_kernel_create(const mfa_attention_kernel_descriptor_t *kernel_descriptor,
                                        mfa_attention_kernel_t **out);
MFA_API void mfa_attention_kernel_destroy(mfa_attention_kernel_t *kernel);

/** kernel.blockDimensions  (:22): out[0..2] = parallelization, traversal, head. */
MFA_API int mfa_attention_kernel_block_dimensions(const mfa_attention_kernel_t *kernel, uint16_t out[3]);
/** kernel.threadgroupSize  (:268-270): threads per CTA of the selected sm_100a kernel. */
MFA_API int mfa_attention_kernel_threadgroup_size(const mfa_attention_kernel_t *kernel, uint32_t *out);
/** kernel.threadgroupMemoryAllocation  (:25, 272-363): dynamic shared memory bytes per CTA. */
MFA_API int mfa_attention_kernel_threadgroup_memory_allocation(const mfa_attention_kernel_t *kernel,
                                                               uint32_t *out);
/** Grid size the dispatch uses: ceil(parallelization dimension / blockDimensions.parallelization)
 *  (SquareAttentionTest.swift:328-339) times batch_count. */
MFA_API int mfa_attention_kernel_grid_size(const mfa_attention_kernel_t *kernel,
                                           const mfa_function_constants_t *constants, uint32_t *out);
/** Name of the compiled kernel family ("attention_forward_tcgen05<128>" ...) -- stands in for
 *  kernel.createSource() (AttentionKernel+Source.swift:11-55), which has no analogue for
 *  ahead-of-time compiled CUDA.  Static storage owned by the kernel handle. */
MFA_API const char *mfa_attention_kernel_source_name(const mfa_attention_kernel_t *kernel);

/** What the reference leaves to its caller: makeLibrary + makeComputePipelineState + setBuffer x10
 *  + dispatchThreadgroups (SquareAttentionTest.swift:240-372).  `buffers[i]` is the DEVICE pointer
 *  bound at AttentionOperand.bufferBinding == i (Q0 K1 V2 O3 L4 D5 dO6 dV7 dK8 dQ9); slots the
 *  kernel type does not touch may be NULL.  Asynchronous on `cuda_stream` (a cudaStream_t, NULL =
 *  default stream).  Kernel order and dependencies are the reference's: forward writes O, L;
 *  backwardQuery reads O, L, dO and writes D, dQ; backwardKeyValue reads L, D and writes dK, dV
 *  (AttentionKernelType.swift:10-22).
 *  Some launches use a library-owned workspace per (device, stream): partial results of grids split across SMs, the
 *  zero-padded staging of head dimensions that are not multiples of 8, the FP16 copy of a BF16 dO.  It grows on demand
 *  with cudaMalloc, which is not possible while `cuda_stream` is being captured into a CUDA graph: encode the same
 *  problem size once outside the capture first (MFA_ERROR_CUDA with that message otherwise). */
MFA_API int mfa_attention_kernel_encode(const mfa_attention_kernel_t *kernel,
                                        const mfa_function_constants_t *constants,
                                        void *const buffers[MFA_BUFFER_COUNT], void *cuda_stream);

/** Number of CUDA kernels one encode() launches (1; +1 when a small grid is split along the traversal axis and a
 *  merge kernel follows: split-KV combine for the forward, a plain sum of partial accumulators for dQ and dK/dV). */
MFA_API int mfa_attention_kernel_launch_count(const mfa_attention_kernel_t *kernel,
                                              const mfa_function_constants_t *constants, uint32_t *out);

/* ------------------------------------------------------------------------------------------ */
/* Kernel cache keyed by descriptor                                                            */
/* ------------------------------------------------------------------------------------------ */
/** The analogue of the reference's pipeline cache (GEMMKernel.register(descriptor:) / pipelineCache[descriptor],
 *  R/GEMM/GEMMDescriptor/GEMMDescriptor+PipelineCache.swift:16-36): descriptor.kernelDescriptor(type:) +
 *  AttentionKernel(descriptor:) run once per distinct (descriptor, type) and the validated kernel object is kept.
 *  R, C and batch_count are launch-time constants and not part of the key.  The returned handle is owned by the
 *  library (do NOT destroy it), is immutable, and stays valid until the process exits.  Thread-safe. */
MFA_API int mfa_attention_kernel_cache_fetch(const mfa_attention_descriptor_t *descriptor, mfa_kernel_type_t type,
                                             const mfa_attention_kernel_t **out);
/** Number of kernel objects the cache currently holds. */
MFA_API int mfa_attention_kernel_cache_size(void);

/* ------------------------------------------------------------------------------------------ */
/* Host-buffer convenience (the e2e path): H2D -> selected kernels -> D2H, synchronous.        */
/* ------------------------------------------------------------------------------------------ */
#define MFA_RUN_FORWARD (1u << MFA_FORWARD)
#define MFA_RUN_BACKWARD_QUERY (1u << MFA_BACKWARD_QUERY)
#define MFA_RUN_BACKWARD_KEY_VALUE (1u << MFA_BACKWARD_KEY_VALUE)

/** `host_buffers[i]` are HOST pointers laid out exactly like the device buffers (element type =
 *  memoryPrecisions[operand]).  Inputs (Q,K,V, and dO for backward) are copied to the device,
 *  the kernels in `run_mask` are encoded in the reference's order fwd -> dQ -> dK/dV, and every
 *  output they produce whose host pointer is non-NULL is copied back.  Device scratch is owned
 *  by the library (grown on demand, one set per calling thread and device).  `device` = CUDA device
 *  ordinal; the caller's current device is restored before the call returns.
 *  With batch_count > 1 the independent problems are processed in chunks that rotate over three
 *  streams, so uploads, kernels and downloads of neighbouring chunks overlap (pass page-locked host
 *  memory to get the overlap; pageable memory still works, serialised by the driver). */
MFA_API int mfa_attention_run_host(const mfa_attention_descriptor_t *descriptor, uint32_t run_mask,
                                   void *const host_buffers[MFA_BUFFER_COUNT], int device);

/* Host-memory placement for the host-buffer path (B200 extension; the reference's buffers are Metal shared-storage
 * buffers, MTLContext+Buffers.swift:5-45, with no placement to speak of on a unified-memory SoC). */
/** Page-locked host buffer for mfa_attention_run_host, allocated (first-touched) on the NUMA node `device` hangs
 *  off and portable across CUDA contexts.  The calling thread's CPU affinity is unchanged on return. */
MFA_API int mfa_host_alloc(size_t bytes, int device, void **out);
/** The same for buffers the host only WRITES and the GPU reads (Q, K, V, dO of mfa_attention_run_host): the pages are also
 *  write-combined, so the upload's PCIe reads are not snooped through the CPU caches and the buffers do not evict the
 *  host's working set.  Reading such a buffer with the CPU is very slow: do not use it for outputs.  Measured
 *  (profiles/r2_e2e_chunks.txt): with upload buffers alone the 201 MB + 135 MB step time is unchanged within the box-to-box
 *  noise (5.7-6.5 ms on that box either way); with the OUTPUT buffers write-combined as well it was 5.10 ms in every run
 *  against 5.3-6.5 ms -- the device-to-host writes into cacheable memory are what the host's cache hierarchy slows down --
 *  but outputs a CPU cannot read at speed are not a configuration this library measures or recommends. */
MFA_API int mfa_host_alloc_upload(size_t bytes, int device, void **out);
MFA_API int mfa_host_free(void *ptr);
/** Restricts the calling thread to the CPUs of `device`'s NUMA node (within the affinity it already has), so that
 *  memory it allocates afterwards and the copies it issues stay on the GPU's socket.  `*numa_node` (optional) receives
 *  the node, or -1 when the platform reports none (then nothing is changed). */
MFA_API int mfa_host_bind_thread_to_device(int device, int *numa_node);

/** Frees what the library holds on `device`: the calling thread's run_host scratch (operand buffers, streams, events)
 *  and every split-grid workspace of the device.  Synchronises the device first.  Optional -- everything is reused
 *  across calls and reclaimed at process exit; long-lived hosts that are done with a device call this. */
MFA_API int mfa_release_device_resources(int device);

/** Element count of operand's buffer for one problem (R*D, C*D, R ...) times batch_count. */
MFA_API int mfa_attention_descriptor_operand_elements(const mfa_attention_descriptor_t *descriptor,
                                                      mfa_operand_t operand, size_t *out);

/* ------------------------------------------------------------------------------------------ */
/* GEMMDescriptor   (R/GEMM/GEMMDescriptor/GEMMDescriptor.swift:10-44)                          */
/* ------------------------------------------------------------------------------------------ */
/* C = A . B, or C += A . B with load_previous_C (AdversarialShapeTest.swift:211-236):
 *   A is M x K (row m at m * lda), or stored K x M when transpose_A (row k at k * lda);
 *   B is K x N (row k at k * ldb), or stored N x K when transpose_B (row n at n * ldb);
 *   C is M x N, row-major, row m at m * ldc.
 * Buffer bindings: A = 0, B = 1, C = 2 (GEMMKernel+Source.swift:42-44). */
#define MFA_GEMM_BUFFER_COUNT 3

typedef struct mfa_gemm_descriptor {
  uint32_t batch_dimension;            /* batchDimension :18.  B200 extension: N > 1 runs N independent problems stored
                                          back to back; problem b of an operand starts at b * trailing * leading
                                          elements (trailing = rows as stored, leading = its leading dimension).  0 = 1. */
  uint8_t has_leading_dimensions;      /* Swift optional `leadingDimensions != nil`   :21 */
  uint8_t load_previous_C;             /* loadPreviousC                                :23 */
  uint8_t has_matrix_dimensions;       /* Swift optional `matrixDimensions != nil`     :37 */
  uint8_t has_memory_precisions;       /* Swift optional `memoryPrecisions != nil`     :39-40 */
  uint8_t has_transpose_state;         /* Swift optional `transposeState != nil`       :42 */
  uint8_t transpose_A, transpose_B;    /* transposeState (A, B) */
  uint8_t memory_precisions[3];        /* memoryPrecisions (A, B, C), mfa_precision_t raw values */
  uint32_t leading_dimensions[3];      /* leadingDimensions (A, B, C) */
  uint32_t M, N, K;                    /* matrixDimensions */
} mfa_gemm_descriptor_t;

/** GEMMDescriptor.init(): batch 1, everything else nil / false. */
MFA_API void mfa_gemm_descriptor_init(mfa_gemm_descriptor_t *descriptor);

/** The launch-time constants: descriptor.setFunctionConstants(_:) (GEMMDescriptor.swift:327-380), indices 0-2 (M, N, K),
 *  5-7 (leading dimensions) and 10 (loadPreviousC), plus the batch extension. */
typedef struct mfa_gemm_function_constants {
  uint32_t M, N, K;
  uint32_t leading_dimensions[3]; /* A, B, C: the descriptor's, or the defaults of chooseLeadingDimension (:340-364) */
  uint8_t load_previous_C;
  uint32_t batch_count;           /* 0/1 = single problem */
} mfa_gemm_function_constants_t;

/** Fills `constants`.  Missing matrixDimensions / transposeState -> MFA_ERROR_INCOMPLETE_DESCRIPTOR ("Descriptor was
 *  incomplete."); a leading dimension below its minimum (K or M for A, N or K for B, N for C) -> MFA_ERROR_INVALID_ARGUMENT
 *  with "Leading block dimension was too small." (:355-357). */
MFA_API int mfa_gemm_descriptor_set_function_constants(const mfa_gemm_descriptor_t *descriptor,
                                                       mfa_gemm_function_constants_t *constants);

/* ------------------------------------------------------------------------------------------ */
/* GEMMKernelDescriptor   (R/GEMM/GEMMKernelDescriptor.swift:21-181)                           */
/* ------------------------------------------------------------------------------------------ */
typedef struct mfa_gemm_kernel_descriptor {
  uint8_t has_block_dimensions;             /* blockDimensions (M, N, K)                       :116 */
  uint16_t block_dimensions[3];
  uint8_t has_leading_block_dimensions;     /* leadingBlockDimensions (A, B, C), optional      :126 */
  uint16_t leading_block_dimensions[3];
  uint8_t has_memory_precisions;            /* memoryPrecisions (A, B, C)                      :128 */
  uint8_t memory_precisions[3];
  uint8_t has_register_precisions;          /* registerPrecisions (A, B, C)                    :165 */
  uint8_t register_precisions[3];
  uint8_t prefer_async_load;                /* preferAsyncLoad: 0 / 1 (default 1)              :139 */
  uint8_t prefer_async_store;               /* preferAsyncStore: 0 / 1 / 0xFF nil              :145 */
  uint8_t has_splits;                       /* splits (M, N)                                   :173 */
  uint16_t splits[2];
  uint8_t has_transpose_state;              /* transposeState (A, B)                           :176 */
  uint8_t transpose_A, transpose_B;
  /* ---- B200 extension: which sm_100a kernel family the heuristic picked ---- */
  uint8_t backend;                          /* mfa_backend_t */
} mfa_gemm_kernel_descriptor_t;

/** GEMMKernelDescriptor.init(): everything nil, preferAsyncLoad true. */
MFA_API void mfa_gemm_kernel_descriptor_init(mfa_gemm_kernel_descriptor_t *kernel_descriptor);

/** GEMMKernelDescriptor(descriptor:)  (GEMMDescriptor.swift:106-234), with this library's heuristic in place of the
 *  Apple one: MFA_BACKEND_TCGEN05 when A and B are both FP16 or both BF16 (any C), MFA_BACKEND_SIMT_FP32 otherwise
 *  (FP32 in A or B, or FP16 beside BF16: tcgen05 kind::f16 cannot mix the two 16-bit types in one MMA, and TF32 would
 *  miss the FP32 tolerance).  Register precisions: A and B keep their memory precision; C is FP32 because both families
 *  accumulate in FP32 (TMEM or registers) -- where the reference picks FP16 for an all-FP16 problem (:196-200).
 *  Missing matrixDimensions / memoryPrecisions / transposeState -> MFA_ERROR_INCOMPLETE_DESCRIPTOR. */
MFA_API int mfa_gemm_descriptor_kernel_descriptor(const mfa_gemm_descriptor_t *descriptor,
                                                  mfa_gemm_kernel_descriptor_t *out);

/* ------------------------------------------------------------------------------------------ */
/* GEMMKernel   (R/GEMM/GEMMKernel/GEMMKernel.swift:10-270)                                     */
/* ------------------------------------------------------------------------------------------ */
typedef struct mfa_gemm_kernel mfa_gemm_kernel_t; /* opaque */

/** GEMMKernel(descriptor:)  (:26-154).  Missing blockDimensions, memoryPrecisions, preferAsyncStore,
 *  registerPrecisions, splits or transposeState -> MFA_ERROR_INCOMPLETE_DESCRIPTOR ("Descriptor was incomplete.").
 *  Register precisions follow the reference's truth table (:46-97): "Operand A had an invalid register precision." (and
 *  B, C) and "BF16 cannot be used as the register precision for C." -> MFA_ERROR_INVALID_PRECISIONS.  An FP16 register
 *  precision for C (legal in the reference) is accepted; the kernels still accumulate in FP32.  Block or leading block
 *  dimensions without a compiled kernel, or a backend the precisions do not fit -> MFA_ERROR_UNSUPPORTED. */
MFA_API int mfa_gemm_kernel_create(const mfa_gemm_kernel_descriptor_t *kernel_descriptor, mfa_gemm_kernel_t **out);
MFA_API void mfa_gemm_kernel_destroy(mfa_gemm_kernel_t *kernel);

/** kernel.blockDimensions (M, N, K) of the compiled kernel  (:21). */
MFA_API int mfa_gemm_kernel_block_dimensions(const mfa_gemm_kernel_t *kernel, uint16_t out[3]);
/** kernel.threadgroupSize  (:260-262): threads per CTA (for tcgen05: 4 epilogue warps + 1 TMA warp + 1 MMA warp). */
MFA_API int mfa_gemm_kernel_threadgroup_size(const mfa_gemm_kernel_t *kernel, uint32_t *out);
/** kernel.threadgroupMemoryAllocation  (:24, 264-269): dynamic shared memory bytes per CTA. */
MFA_API int mfa_gemm_kernel_threadgroup_memory_allocation(const mfa_gemm_kernel_t *kernel, uint32_t *out);
/** Output tiles of the dispatch: ceil(N / block N) * ceil(M / block M) * batch (AdversarialShapeTest.swift:152-158).
 *  The tcgen05 kernel is persistent: it launches min(tiles, SM count) CTAs that loop over these tiles. */
MFA_API int mfa_gemm_kernel_grid_size(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *constants,
                                      uint32_t *out);
/** CUDA kernels one encode() launches: 1, plus (tcgen05) one staging copy per 16-bit operand whose leading dimension is
 *  not a multiple of 8 elements.  A base pointer that is not 16-byte aligned also stages its operand (one more launch,
 *  which the constants alone cannot predict). */
MFA_API int mfa_gemm_kernel_launch_count(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *constants,
                                         uint32_t *out);
/** Name of the compiled kernel ("gemm_tcgen05<bfloat, bfloat, float, NN>" ...), standing in for createSource(). */
MFA_API const char *mfa_gemm_kernel_source_name(const mfa_gemm_kernel_t *kernel);

/** Binds A, B, C (device pointers, bindings 0, 1, 2) and dispatches on `cuda_stream` (NULL = default stream) of the
 *  current device; asynchronous.  C may alias nothing else; with load_previous_C it is read and written in place.
 *  The staging copies of the tcgen05 family use a library-owned workspace per (device, stream), which grows with
 *  cudaMalloc: encode the same problem once outside a CUDA-graph capture before capturing it.
 *  No sm_100 device -> MFA_ERROR_NO_DEVICE (no CPU fallback). */
MFA_API int mfa_gemm_kernel_encode(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *constants,
                                   void *const buffers[MFA_GEMM_BUFFER_COUNT], void *cuda_stream);

/** GEMMKernel.register(descriptor:) + pipelineCache[descriptor] (GEMMDescriptor+PipelineCache.swift:16-36): the
 *  kernel object of the descriptor, created once.  The key is what the kernel descriptor depends on -- memory
 *  precisions and transposes; M, N, K, the leading dimensions, load_previous_C and the batch are launch constants.  The
 *  handle is owned by the library (do NOT destroy it), immutable and valid until process exit.  Thread-safe. */
MFA_API int mfa_gemm_kernel_cache_fetch(const mfa_gemm_descriptor_t *descriptor, const mfa_gemm_kernel_t **out);
/** Number of GEMM kernel objects the cache holds. */
MFA_API int mfa_gemm_kernel_cache_size(void);

#ifdef __cplusplus
} /* extern "C" */
#endif
#endif /* MFA_B200_H */
